"""The Metropolis chain on the wide path (32 < d <= 256 parameters: a truncated KL prior whose parameter
vector lives in shared memory): a recomputed Phi(u), runs split over several launches, and the largest
parameter vector."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


def _kl_problem(G, N, m, numerics):
    """A KL-prior Burgers problem with m modes; data from a truth that excites the modes."""
    import ip_mcmc_b200 as M
    f = M.BurgersFVM(N=N, kl_modes=m, numerics=numerics)
    lam = np.concatenate([np.full(3, 0.25 ** 2), M.BurgersFVM.kl_prior_variances(m, scale=0.05)])
    rng = np.random.default_rng(m)
    truth = np.concatenate([G.TRUTH, 0.3 * np.sqrt(lam[3:]) * rng.standard_normal(m)])
    pot = M.EvolutionPotential(f, f.at_parameters(truth), M.GaussianDistribution(np.zeros(5), G.NOISE_COV))
    return f, pot, lam


def _pcn(d, lam, beta=0.2, **kw):
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    return M.SamplerSpec(d, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta,
                         factor=np.sqrt(lam), **kw)


def _boxed_rw(d, lam, delta=0.02, **kw):
    """RW with the prior regulariser and a box on the shock position (component 2)."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    m = d - 3
    box = M.BoxConstraint(np.r_[-np.inf, -np.inf, -0.62, np.full(m, -np.inf)],
                          np.r_[np.inf, np.inf, -0.38, np.full(m, np.inf)], shift=np.r_[0, 0, -0.5, np.zeros(m)])
    return M.SamplerSpec(d, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * delta),
                         factor=np.sqrt(lam), prior_chol=np.diag(np.sqrt(lam)), constraint=box, **kw)


@pytest.mark.parametrize("numerics", ["exact", "fused"])
def test_wide_recompute_phi_u_is_bit_equivalent(G, numerics):
    """Solving for Phi(u) again every step (the reference's two solves per step) gives the same chain as
    carrying it: same states and step-log Phi(v), a, decisions; one more solve per step."""
    d = 3 + 61
    f, pot, lam = _kl_problem(G, 128, 61, numerics)
    n = 20
    rng = np.random.default_rng(4)
    w = rng.standard_normal((n, d)) * np.sqrt(lam)
    U = rng.random(n)
    s1, l1, v1, c1 = G.run_injected(pot, _pcn(d, lam), np.zeros(d), w, U, n_copies=3)
    s2, l2, v2, c2 = G.run_injected(pot, _pcn(d, lam, recompute_phi_u=True), np.zeros(d), w, U, n_copies=3)
    assert np.array_equal(s1, s2) and np.array_equal(v1, v2) and np.array_equal(l1[..., :3], l2[..., :3])
    assert 0 < c1.counters[0, 1].item() < n
    assert c1.counters[:, 3].tolist() == [n + 1] * 3
    assert c2.counters[:, 3].tolist() == [2 * n + 1] * 3
    assert torch.equal(c1.counters[:, [0, 1, 4, 5]], c2.counters[:, [0, 1, 4, 5]])


def _run_split(pot, spec, d, n_chains, total, per_launch):
    """`total` steps of free-running chains in launches of `per_launch` steps; returns the recorded trace
    (burn-in and thinning from `spec`) and the chain batch."""
    import ip_mcmc_b200 as M

    def recorded_before(g):
        return max(0, g - spec.record_start) // spec.record_interval

    ch = M.ChainBatch(pot.problem(), np.zeros(d), n_chains=n_chains)
    parts = []
    for g0 in range(0, total, per_launch):
        g1 = min(total, g0 + per_launch)
        k = recorded_before(g1) - recorded_before(g0)
        tr = torch.empty((n_chains, k, d), dtype=torch.float64, device="cuda") if k else None
        ch.run(spec, g1 - g0, trace=tr)
        if tr is not None:
            parts.append(tr)
    return torch.cat(parts, dim=1).cpu().numpy(), ch


@pytest.mark.parametrize("kind", ["pcn", "boxed_rw"])
def test_wide_split_launches_match_one_launch(G, kind):
    """A run split over launches of 7 steps reloads u, Phi(u) and the moments, recomputes the prior regulariser
    of u, and accumulates counters and moments: everything must equal one launch of all steps bit for bit."""
    d, total, n_chains = 3 + 61, 30, 40
    f, pot, lam = _kl_problem(G, 128, 61, "fused")
    spec = (_pcn if kind == "pcn" else _boxed_rw)(d, lam, seed=11, record_start=4, record_interval=3)
    one, a = _run_split(pot, spec, d, n_chains, total, total)
    split, b = _run_split(pot, spec, d, n_chains, total, 7)
    assert a.launches == 1 and b.launches == 5
    assert one.shape == (n_chains, 8, d) and np.array_equal(one, split)
    for name in ("u", "phi", "counters", "mom_count", "mom_mean", "mom_m2"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(a.pooled(), b.pooled())
    cnt = a.counters.cpu().numpy()
    assert np.all(cnt[:, 0] == total) and 0 < cnt[:, 1].sum() < n_chains * total
    assert np.all(cnt[:, 3] + cnt[:, 5] == total + 1)            # a solve per step inside the box, plus Phi(u_0)
    assert (cnt[:, 5].sum() > 0) == (kind == "boxed_rw")
    assert np.all(a.mom_count.cpu().numpy() == 8)


def test_wide_largest_parameter_vector(G):
    """d = 256 (253 KL modes), the largest wide vector: free-running pCN chains run and count every step."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    d, n, n_chains = 256, 12, 20
    assert d == _lib.MAX_DIM_WIDE
    f, pot, lam = _kl_problem(G, 128, d - 3, "fused")
    ch = M.ChainBatch(pot.problem(), np.zeros(d), n_chains=n_chains)
    trace = torch.empty((n_chains, n, d), dtype=torch.float64, device="cuda")
    ch.run(_pcn(d, lam, seed=5), n, trace=trace)
    tr = trace.cpu().numpy()
    assert tr.shape == (n_chains, n, d) and np.all(np.isfinite(tr)) and torch.isfinite(ch.phi).all()
    cnt = ch.counters.cpu().numpy()
    assert np.all(cnt[:, 0] == n) and np.all(cnt[:, 3] == n + 1) and np.all(cnt[:, 4] == 0) and np.all(cnt[:, 5] == 0)
    assert 0 < cnt[:, 1].sum() < n_chains * n
    assert np.array_equal(ch.u.cpu().numpy(), tr[:, -1])
    np.testing.assert_allclose(ch.mom_mean.cpu().numpy(), tr.mean(1), rtol=1e-12, atol=1e-15)
