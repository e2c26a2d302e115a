"""GPU parity of the Lorenz-96 path.  Parity is pinned at the RHS (bit-exact), the single
Dormand-Prince attempt and short horizons; over T = 20 any two roundings of the same algorithm
diverge (positive Lyapunov exponent), so long solves are compared statistically (SURVEY.md
section 7 'Lorenz chaos')."""
import functools

import numpy as np
import pytest
import torch

from conftest import golden
from oracle import lorenz_np as L
from oracle import mcmc_np as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


# (K, J) beside the reference's (6, 4): with it, every compiled kernel variant (<J, K = 6 or run-time K>) and every way a
# warp splits into lane groups of K lanes -- 10 groups and 2 idle lanes (K = 3), full warps with the shared-memory slot of
# idle lanes unused (K = 4, 8), 2 groups with 10 / 8 idle lanes (K = 11, 12) -- and J = 1 (the fast block mean of one
# variable) and J = 8 (pairwise block mean, 9 values per lane)
LORENZ_GRID = [(3, 1), (4, 2), (5, 8), (6, 2), (7, 4), (8, 4), (11, 2), (12, 8)]
LORENZ_THETA = np.array([10.0, 10.0, 10.0])      # (F, h, b) of the reference, c = 1 (lorenz_mcmc.py:91)


@functools.lru_cache(maxsize=None)
def _lorenz_problem(K, J):
    """An inverse problem at any (K, J), in the layout of tests/golden/lorenz_problem_K6_J4.npz: a seeded random state
    spun up for 2 time units with the oracle's solver, data = the oracle's G at a truth (T = 0.5), and the variances
    of a diagonal noise covariance."""
    rng = np.random.default_rng(1000 * K + J)
    spin = L.LorenzProblem(K, J, 2.0, 1, LORENZ_THETA, rng.standard_normal(K * (J + 1)))
    spin(np.zeros(3))
    ic = spin.IC.copy()
    y = L.LorenzProblem(K, J, 0.5, 1, LORENZ_THETA, ic)(np.array([0.5, -0.5, 0.5]))
    return dict(prior_means=LORENZ_THETA, IC=ic, y=y, var=1.0 + y ** 2, u0=np.array([-0.5, 0.9, 0.2]))


def _lorenz_setup(T, p=None, numerics="exact", K=6, J=4):
    import ip_mcmc_b200 as M
    if p is None:
        p = golden("lorenz_problem_K6_J4.npz") if (K, J) == (6, 4) else _lorenz_problem(K, J)
    f = M.Lorenz96Moments(K, J, T, 1, p["prior_means"], p["IC"], numerics=numerics)
    noise = M.GaussianDistribution(np.zeros(5 * K), 0.5 ** 2 * np.diag(p["var"]))     # lorenz_mcmc.py:111-112
    prior = M.GaussianDistribution(np.zeros(3), np.diag([10., 1, 10]))            # lorenz_mcmc.py:115,119
    pot = M.EvolutionPotential(f, p["y"], noise)
    return f, pot, prior, p


def test_rhs_bit_identical_to_reference(G):
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    g = golden("lorenz_rhs.npz")
    for i in range(int(g["n_cases"])):
        K, J = int(g[f"case{i}_K"]), int(g[f"case{i}_J"])
        n = 11          # more states than fit one warp: exercises group packing and the tail
        th = G.cuda(np.tile([float(g[f"case{i}_{k}"]) for k in "Fhcb"], (n, 1)))
        st = G.cuda(np.tile(g[f"case{i}_state"], (n, 1)))
        out = torch.empty_like(st)
        _lib.check(lib.ipmcmc_lorenz_rhs(K, J, 0, n, th.data_ptr(), st.data_ptr(), out.data_ptr(), None))
        o = out.cpu().numpy()
        assert all(np.array_equal(o[k], g[f"case{i}_rhs"]) for k in range(n)), (K, J)


def test_reference_rhs_known_answers(G):
    """lorenz.py:114-147 (K >= 1 supported by the probe)."""
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    cases = [((4, 1), (0, 0, 0, 0), [1, 2, 3, 4, 0, 0, 0, 0], [-5, -3, 3, -7, 0, 0, 0, 0]),
             ((1, 4), (0, 0, 1, 2), [0, 1, 2, 3, 4], [0, 3, -20, 5, -2]),
             ((1, 2), (0, 2, -1, 0), [0, 1, 2], [3, 1, 2]),
             ((2, 2), (1, 1, 1, 1), [2, 3, 4, 5, 6, 7], [-2.5, -10.5, 2, -8, 2.5, -11.5]),
             ((3, 1), (2, 1, 1, 1), [0, 0, 0, 0, 0, 0], [2, 2, 2, 0, 0, 0])]
    for (K, J), th, s, want in cases:
        for num in (0, 1):                        # exact and fused numerics (small integers: both exact)
            tht, st = G.cuda([th]), G.cuda([s])
            out = torch.empty_like(st)
            _lib.check(lib.ipmcmc_lorenz_rhs(K, J, num, 1, tht.data_ptr(), st.data_ptr(), out.data_ptr(), None))
            np.testing.assert_allclose(out.cpu().numpy()[0], want, rtol=1e-15, atol=1e-15)


def test_fused_rhs_close_to_reference(G):
    """FUSED numerics contract the right-hand side (FMAs, factored products): same function, a
    few ulps of the largest term away from the reference's rounding order."""
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    g = golden("lorenz_rhs.npz")
    for i in range(int(g["n_cases"])):
        K, J = int(g[f"case{i}_K"]), int(g[f"case{i}_J"])
        n = 7
        th = G.cuda(np.tile([float(g[f"case{i}_{k}"]) for k in "Fhcb"], (n, 1)))
        st = G.cuda(np.tile(g[f"case{i}_state"], (n, 1)))
        out = torch.empty_like(st)
        _lib.check(lib.ipmcmc_lorenz_rhs(K, J, 1, n, th.data_ptr(), st.data_ptr(), out.data_ptr(), None))
        o = out.cpu().numpy()
        ref = g[f"case{i}_rhs"]
        scale = max(1.0, float(np.abs(g[f"case{i}_state"]).max()) ** 2 * 12)     # size of the largest term
        for k in range(n):
            np.testing.assert_allclose(o[k], ref, rtol=1e-13, atol=1e-14 * scale)


def _kj_params(extra, reference_ids):
    """pytest parameters (K, J) + extra over the reference's (6, 4), whose ids stay `reference_ids`, and LORENZ_GRID."""
    out = [pytest.param(6, 4, *e, id=i) for e, i in zip(extra, reference_ids)]
    out += [pytest.param(K, J, *e, id="K%dJ%d-%s" % (K, J, i)) for K, J in LORENZ_GRID for e, i in zip(extra, reference_ids)]
    return out


@pytest.mark.parametrize("K,J,num", _kj_params([(0,), (1,)], ["0", "1"]))
def test_single_rk45_attempt_vs_scipy_restatement(G, K, J, num):
    """One Dormand-Prince attempt: y_new, f_new and the RMS error norm against oracle/lorenz_np.py
    (bit-identical to scipy).  Device stage sums are FMA chains, scipy's are BLAS dots: agreement
    to 1e-12 relative (north_star 1e-10).  The error norm is a sum over the chain's K lanes: at K != 6 the
    run-time-K shuffle tree of LorenzLanes::group_sum."""
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    p = golden("lorenz_problem_K6_J4.npz") if (K, J) == (6, 4) else _lorenz_problem(K, J)
    nv = K * (J + 1)
    rng = np.random.default_rng(4)
    n = 13
    thetas = np.column_stack([rng.uniform(8, 12, n), rng.uniform(8, 12, n), np.ones(n), rng.uniform(8, 12, n)])
    states = p["IC"] + 0.1 * rng.standard_normal((n, nv))
    # the grid's states rest near the fixed point of the J <= 2 systems, where steps below 1e-2 give error norms of
    # ~1e-9: the cancellation of much larger stage terms, on which no two summation orders agree to 1e-9
    hs = 10 ** rng.uniform(-3 if (K, J) == (6, 4) else -2, -1.3, n)
    out = torch.empty((n, 2 * nv + 1), dtype=torch.float64, device="cuda")
    tht, st, ht = G.cuda(thetas), G.cuda(states), G.cuda(hs)
    _lib.check(lib.ipmcmc_lorenz_rk45_attempt(K, J, num, n, tht.data_ptr(), st.data_ptr(), ht.data_ptr(), 1e-3, 1e-6,
                                              out.data_ptr(), None))
    o = out.cpu().numpy()
    for i in range(n):
        fun = lambda t, s: L.lorenz_rhs(s, K, J, *thetas[i])
        yn, fn, err, _ = L.rk45_attempt(fun, 0.0, states[i], fun(0, states[i]), hs[i])
        np.testing.assert_allclose(o[i, :nv], yn, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(o[i, nv:2 * nv], fn, rtol=1e-10, atol=1e-11)
        np.testing.assert_allclose(o[i, 2 * nv], err, rtol=1e-9)


@pytest.mark.parametrize("numerics", ["exact", "fused"])
def test_short_solves_vs_reference(G, numerics):
    """solve_ivp parity while chaos has not yet amplified rounding: same accepted/rejected step
    counts (controller decisions) and G / end state close to the reference's."""
    gs = golden("lorenz_solves.npz")
    for i in range(int(gs["n_cases"])):
        T = float(gs[f"case{i}_T"])
        if T > 2:
            continue
        f, pot, _, p = _lorenz_setup(T, numerics=numerics)
        r = f.batch(gs[f"case{i}_u"].reshape(1, 3), p["IC"].reshape(1, -1))
        acc, rej = r["work"][0].tolist()
        assert acc == int(gs[f"case{i}_n_t"]) - 1
        assert 2 + 6 * (acc + rej) == int(gs[f"case{i}_nfev"])
        tol = {0.25: 1e-11, 1.0: 1e-8, 2.0: 1e-4}[T]       # e^(lambda T) growth of 1e-16 seeds
        np.testing.assert_allclose(r["G"].cpu().numpy()[0], gs[f"case{i}_G"], rtol=tol, atol=tol)
        np.testing.assert_allclose(r["state"].cpu().numpy()[0], gs[f"case{i}_IC_end"], rtol=0, atol=100 * tol)


@pytest.mark.parametrize("numerics", ["exact", "fused"])
def test_short_solves_over_the_lane_group_grid(G, numerics):
    """Forward solves at every (K, J) of LORENZ_GRID against the oracle's solve_ivp restatement, T = 0.25 and 1,
    over batches that leave the last lane group of a warp partly empty: the same accepted and rejected RK45
    attempts (controller decisions, each resting on a group-summed error norm), G and the end state within the
    tolerances of test_short_solves_vs_reference.  Somewhere on the grid the controller rejects attempts."""
    rejected = 0
    for K, J in LORENZ_GRID:
        p = _lorenz_problem(K, J)
        groups = 32 // K
        n = 2 * groups - 1 if groups <= 4 else groups + 1          # never a multiple of the chains per warp
        rng = np.random.default_rng(10 * K + J)
        us = rng.uniform(-1, 1, (n, 3))
        # started off the attractor (a fixed point for J <= 2): near it the error norms of the controller are
        # cancellation-dominated and the step sizes of two implementations part at 1e-9
        ics = p["IC"] + rng.standard_normal((n, K * (J + 1)))
        for T, tol in ((0.25, 1e-11), (1.0, 1e-8)):
            f, _, _, _ = _lorenz_setup(T, numerics=numerics, K=K, J=J)
            r = f.batch(us, ics)
            Gd, st, work = r["G"].cpu().numpy(), r["state"].cpu().numpy(), r["work"].cpu().numpy()
            for i in range(n):
                op = L.LorenzProblem(K, J, T, 1, p["prior_means"], ics[i])
                g_ref = op(us[i])
                assert (work[i, 0], work[i, 1]) == (op.n_accepted, op.n_rejected), (K, J, T, i)
                np.testing.assert_allclose(Gd[i], g_ref, rtol=tol, atol=tol, err_msg=str((K, J, T, i)))
                np.testing.assert_allclose(st[i], op.IC, rtol=0, atol=100 * tol, err_msg=str((K, J, T, i)))
                rejected += op.n_rejected
    assert rejected > 0


@pytest.mark.parametrize("numerics", ["exact", "fused"])
@pytest.mark.parametrize("c", [1.0, 3.0])
def test_short_solves_other_time_scale_ratio_and_small_b(G, numerics, c):
    """FUSED integrates the scaled fast variables Z = -b c Y and specialises c = 1 (the reference's value): the
    general-c code path, and parameters with b close to zero (scale clamped at 1e-30, a linear fast system), against
    the oracle's solve_ivp restatement: same step counts, G and end state to 1e-9."""
    import ip_mcmc_b200 as M
    p = golden("lorenz_problem_K6_J4.npz")
    T = 0.25
    us = [np.array([-1.9, 1.9, 0.9]), np.array([0.5, -2.0, -3.0]),
          -p["prior_means"] + np.array([9.0, 8.0, 1e-9]),      # b = 1e-9
          -p["prior_means"] + np.array([11.0, 9.0, 0.0])]      # b = 0: the quadratic term vanishes
    for u in us:
        f = M.Lorenz96Moments(6, 4, T, c, p["prior_means"], p["IC"], numerics=numerics)
        op = L.LorenzProblem(6, 4, T, c, p["prior_means"], p["IC"])
        r = f.batch(u.reshape(1, 3), p["IC"].reshape(1, -1))
        g_ref = op(u)
        acc, rej = r["work"][0].tolist()
        assert (acc, rej) == (op.n_accepted, op.n_rejected), (c, u)
        np.testing.assert_allclose(r["G"].cpu().numpy()[0], g_ref, rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(r["state"].cpu().numpy()[0], op.IC, rtol=0, atol=1e-8)


def test_stateful_operator_and_potential_semantics(G):
    """LorenzObservationOperator carries its IC (lorenz_mcmc.py:66): two successive calls differ
    and equal one solve continued from the first end state; Phi matches the oracle's logpdf."""
    f, pot, _, p = _lorenz_setup(0.25)
    u = np.array([-1.9, 1.9, 0.9])
    op = L.LorenzProblem(6, 4, 0.25, 1, p["prior_means"], p["IC"])
    opot = O.Potential(op, p["y"], 0.25 * np.diag(p["var"]))
    for _ in range(3):
        g_dev, g_ref = f(u), op(u)
        np.testing.assert_allclose(g_dev, g_ref, rtol=1e-9)
        np.testing.assert_allclose(f.IC, op.IC, rtol=0, atol=1e-9)
    f2, pot2, _, _ = _lorenz_setup(0.25)
    op2 = L.LorenzProblem(6, 4, 0.25, 1, p["prior_means"], p["IC"])
    opot2 = O.Potential(op2, p["y"], 0.25 * np.diag(p["var"]))
    for _ in range(2):
        np.testing.assert_allclose(pot2(u), opot2(u), rtol=1e-9)


@pytest.mark.parametrize("numerics", ["exact", "fused"])
def test_long_solves_statistically(G, numerics):
    """T = 20 (the reference's setting): G(u) is a noisy time average; device and reference
    realisations must agree within the natural variability, and step counts within a few %.
    FUSED is what bench.py measures."""
    gs = golden("lorenz_solves.npz")
    for i in range(int(gs["n_cases"])):
        T = float(gs[f"case{i}_T"])
        if T < 20:
            continue
        f, pot, _, p = _lorenz_setup(T, numerics=numerics)
        n = 64
        ic = p["IC"] + 1e-9 * np.random.default_rng(i).standard_normal((n, 30))   # decorrelated realisations
        r = f.batch(np.tile(gs[f"case{i}_u"], (n, 1)), ic)
        Gd = r["G"].cpu().numpy()
        sd = Gd.std(0) + 1e-12
        z = np.abs(gs[f"case{i}_G"] - Gd.mean(0)) / sd
        assert np.all(z < 5), z.max()        # the reference realisation is a typical member
        acc = r["work"][:, 0].double().mean().item()
        assert abs(acc - (int(gs[f"case{i}_n_t"]) - 1)) < 0.08 * acc


def test_lorenz_chain_first_steps_and_statistics(G):
    """Reference chain (pCN beta=0.5, T=2) replayed with injected noise: proposals are bit-identical
    while decisions agree; Phi of the first step agrees closely (before chaos decorrelates the
    carried IC).  Then free-running chains: acceptance in the reference's ballpark."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    g = golden("chain_lorenz_pcn_T2.npz")
    f, pot, prior, p = _lorenz_setup(float(g["T"]))
    beta = float(g["beta"])
    spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta,
                         recompute_phi_u=True)
    states, slog, vlog, ch = G.run_injected(pot, spec, g["u0"], g["normals"], g["uniforms"], n_copies=7)
    assert np.all(states == states[0]) and np.all(slog == slog[0])        # lanes groups agree
    assert np.array_equal(vlog[0, 0], g["v"][0])
    # Phi(v) of step 1 is the SECOND solve (after Phi(u)): 4 time units of chaotic growth on 1e-16 seeds
    np.testing.assert_allclose(slog[0, 0, 0], g["phi_v"][0], rtol=5e-2)
    same = np.cumprod(np.all(states[0] == g["samples"], axis=1)).sum()
    assert same >= 1          # identical decisions until chaos flips a borderline accept
    # free-running: 2 solves per step (Phi(u) then Phi(v)), counters consistent
    s = M.MCMCSampler(M.ConstSteppCNProposer(beta, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(1))
    out = s.run(g["u0"], 30, 0, 1, n_chains=33)
    assert out.shape == (33, 30, 3)
    acc = s.accepter.ratio()
    assert 0.25 < acc < 0.9, acc          # reference: 24/40 at T=2, "around 0.6" at T=20 (lorenz.org:277-279)
    assert s.last_run["counters"]["work_a"] > 33 * 30 * 2 * 50


@pytest.mark.parametrize("K,J,n_chains,n_samples,steps_per_launch",
                         [pytest.param(6, 4, 33, 6, None, id="33-6-None"), pytest.param(6, 4, 1003, 5, 2, id="1003-5-2"),
                          pytest.param(6, 4, 7, 4, 3, id="7-4-3"),
                          pytest.param(3, 1, 7003, 3, 2, id="K3J1-7003-3-2"), pytest.param(4, 2, 6007, 3, 2, id="K4J2-6007-3-2")])
def test_lorenz_queue_is_pure_scheduling(G, K, J, n_chains, n_samples, steps_per_launch, monkeypatch):
    """The dynamic step scheduler of the Lorenz kernel (work unit = a warp's group of 32 // K chains, the carried
    initial condition travelling through L2 between work items) is pure scheduling: samples, carried
    states, counters and moments are the same bits with one step per work item in one launch and with three
    steps per item over the launch split (ragged last group, several launches, more groups than SMs).  At K = 3
    and K = 4 the batches fit one wave, but the CTA shared memory caps the warps per CTA below ceil(warps / n_SM),
    so the launch has more CTAs than SMs (engine.cu, run_chains)."""
    import ip_mcmc_b200 as M
    groups = 32 // K
    warps = -(-n_chains // groups)
    if K != 6:
        n_sm = torch.cuda.get_device_properties(0).multi_processor_count
        fit = (48 * 1024) // ((groups + 1) * 2 * 64 * 8)                  # lorenz_warps_fit
        assert warps <= 8 * n_sm and -(-warps // n_sm) > fit and -(-warps // fit) > n_sm, (warps, fit, n_sm)
    f, pot, prior, p = _lorenz_setup(0.5, numerics="fused", K=K, J=J)
    mk = lambda: M.MCMCSampler(M.ConstStepStandardRWProposer(0.125, prior),
                               M.CountedAccepter(M.StandardRWAccepter(pot, prior)), np.random.default_rng(5))
    a, b = mk(), mk()
    out_a = a.run(p["u0"], n_samples, 2, 1, n_chains=n_chains)
    monkeypatch.setenv("IPMCMC_SCHED_CHUNK", "3")
    out_b = b.run(p["u0"], n_samples, 2, 1, n_chains=n_chains, steps_per_launch=steps_per_launch)
    ca, cb = a.last_run["chains"], b.last_run["chains"]
    assert ca.sched is not None and cb.sched is not None
    assert np.array_equal(out_a, out_b)
    assert torch.equal(ca.model_state, cb.model_state)
    assert torch.equal(ca.counters, cb.counters) and torch.equal(ca.u, cb.u) and torch.equal(ca.phi, cb.phi)
    assert torch.equal(ca.mom_count, cb.mom_count) and torch.equal(ca.mom_mean, cb.mom_mean) and torch.equal(ca.mom_m2, cb.mom_m2)
    assert a.accepter.calls == b.accepter.calls and a.accepter.accepts == b.accepter.accepts


def test_lorenz_host_entry_point_matches_device_path(G):
    """MCMCSampler.run_host (ipmcmc_sample_host: host buffers, copies inside the C call) == MCMCSampler.run on Lorenz
    chains of a run-time-K kernel: samples, counters, final states and potentials, carried model states."""
    import ip_mcmc_b200 as M
    f, pot, prior, p = _lorenz_setup(0.25, numerics="fused", K=7, J=4)
    mk = lambda: M.MCMCSampler(M.ConstStepStandardRWProposer(0.125, prior),
                               M.CountedAccepter(M.StandardRWAccepter(pot, prior)), np.random.default_rng(8))
    s, h = mk(), mk()
    ref = s.run(p["u0"], 5, 0, 1, n_chains=9)
    got = h.run_host(p["u0"], 5, 0, 1, n_chains=9)
    assert h.last_run["seed"] == s.last_run["seed"]
    assert np.array_equal(got, ref)
    assert np.array_equal(h.last_run["per_chain_counters"], s.last_run["per_chain_counters"].cpu().numpy())
    assert h.accepter.calls == 45 and h.accepter.accepts == s.accepter.accepts
    assert np.array_equal(h.last_run["u"], s.last_run["u"].cpu().numpy())
    assert np.array_equal(h.last_run["phi"], s.last_run["phi"].cpu().numpy())
    assert np.array_equal(h.last_run["model_state"], s.last_run["chains"].model_state.cpu().numpy())


def test_lorenz_library_allocates_queue_scratch(G):
    """ipmcmc_run without scheduler scratch (sched_dev = NULL) on Lorenz chains: the same bits, carried states
    included, as with ChainBatch's scratch."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    f, pot, prior, p = _lorenz_setup(0.5, numerics="fused")
    spec = M.SamplerSpec(3, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=0.5, factor=np.sqrt([10., 1, 10]),
                         prior_chol=prior.L, recompute_phi_u=True, seed=11)
    runs = []
    for own in (True, False):
        ch = M.ChainBatch(pot.problem(), p["u0"], n_chains=23)
        assert ch.sched is not None
        if not own:
            ch.sched = None
        trace = torch.empty((23, 4, 3), dtype=torch.float64, device="cuda")
        ch.run(spec, 4, trace=trace)
        runs.append((trace, ch))
    (ta, ca), (tb, cb) = runs
    assert torch.equal(ta, tb)
    for name in ("model_state", "u", "phi", "counters", "mom_count", "mom_mean", "mom_m2"):
        assert torch.equal(getattr(ca, name), getattr(cb, name)), name


@pytest.mark.parametrize("numerics", ["exact", "fused"])
@pytest.mark.parametrize("K,J,n_chains", [pytest.param(6, 4, 7, id="7"), pytest.param(6, 4, 13, id="13")]
                         + [pytest.param(K, J, 32 // K + 1, id="K%dJ%d" % (K, J)) for K, J in LORENZ_GRID])
def test_lorenz_box_constraint_matches_oracle(G, K, J, n_chains, numerics):
    """ConstrainAccepter on the Lorenz kernels: K = 6 leaves lanes 30, 31 of every warp without a chain and
    n_chains is not a multiple of the 5 chains a warp holds, so the warp-wide ballot of the box test runs
    with idle lanes and an idle tail group (all 32 lanes must take part, lorenz_kernels.cuh).  The other (K, J)
    run one full warp and a tail group of one chain.  Injected noise; compared with the oracle chain: a violated
    box rejects without consuming a uniform and without a solve (accepter.py:52-55), every other decision and
    state equal."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    T, n_steps, delta = 0.05, 12, 0.3      # 24 carried solves = 1.2 time units: rounding differences stay ~1e-8
    f, pot, prior, p = _lorenz_setup(T, numerics=numerics, K=K, J=J)
    lo, hi = -1.0, 1.3
    box = M.BoxConstraint([-np.inf, lo, -np.inf], [np.inf, hi, np.inf], shift=[0.0, 0.0, 0.0])
    rng = np.random.default_rng(21)
    u0 = np.array([-0.5, 0.9, 0.2])
    normals = rng.standard_normal((n_chains, n_steps, 3)) * np.sqrt([10., 1, 10])
    spec = M.SamplerSpec(3, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * delta), prior_chol=prior.L,
                         constraint=box, recompute_phi_u=True)
    # oracle chains first: they tell which steps consume a uniform
    U_dev = np.full((n_chains, n_steps), 0.5)
    refs = []
    for c in range(n_chains):
        op = L.LorenzProblem(K, J, T, 1, p["prior_means"], p["IC"])
        opot = O.Potential(op, p["y"], 0.25 * np.diag(p["var"]))
        tape = rng.random(n_steps)
        ref = O.run_chain(opot, u0, normals[c], tape, O.RW, O.RW, delta, prior_cov=np.diag([10., 1, 10]),
                          constraint=lambda v: lo < v[1] < hi, recompute_phi_u=True)
        valid = ~np.isnan(ref["a"])
        U_dev[c, valid] = tape[:valid.sum()]
        refs.append((ref, valid, op))
    ch = M.ChainBatch(pot.problem(), u0, n_chains=n_chains)
    trace = torch.empty((n_chains, n_steps, 3), dtype=torch.float64, device="cuda")
    slog = torch.empty((n_chains, n_steps, 4), dtype=torch.float64, device="cuda")
    ch.run(spec, n_steps, trace=trace, steplog=slog, inject_w=G.cuda(normals), inject_u=G.cuda(U_dev))
    states, sl, cnt = trace.cpu().numpy(), slog.cpu().numpy(), ch.counters.cpu().numpy()
    n_viol = 0
    for c, (ref, valid, op) in enumerate(refs):
        assert np.array_equal(states[c], ref["u"]), c
        assert cnt[c, 0] == n_steps and cnt[c, 1] == ref["accepts"] and cnt[c, 5] == (~valid).sum()
        assert cnt[c, 2] + cnt[c, 3] == op.n_accepted + op.n_rejected        # no solve on constrained steps
        np.testing.assert_allclose(sl[c, valid, 0], ref["phi_v"][valid], rtol=1e-6)
        assert np.all(np.isnan(sl[c, ~valid, 0]))
        n_viol += (~valid).sum()
    assert n_viol > 0.1 * n_chains * n_steps                                  # the box actually triggers
