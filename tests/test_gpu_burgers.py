"""GPU parity of the Burgers path against the reference-generated fixtures (tests/golden) and the
CPU oracle.  EXACT numerics: bit-identical (stronger than north_star's 1e-10 relative);
FUSED numerics: <= 1e-10 relative (tolerance stated in BASELINE.json north_star)."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import burgers_np as B
from oracle import mcmc_np as O

pytestmark = pytest.mark.gpu
RTOL = 1e-10      # north_star: "match the reference to 1e-10 relative in fp64"


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


@pytest.mark.parametrize("N", [32, 64, 100, 128, 200, 256, 1024])
def test_forward_exact_is_bit_identical_to_reference(G, N):
    g = golden(f"burgers_forward_N{N}.npz")
    f, pot, _, _ = G.burgers_setup(N, "exact", y=g["y"])
    assert np.array_equal(f.x, g["x"]) and f.dx == g["dx"] and f.dx_meas == g["dx_meas"]
    assert np.array_equal(f.left_limits, g["left"]) and np.array_equal(f.right_limits, g["right"])
    r = pot.problem().forward(g["u"], want_state=True)
    assert np.array_equal(r["state"].cpu().numpy(), g["end_state"])
    assert np.array_equal(r["G"].cpu().numpy(), g["G"])
    assert np.array_equal(r["phi"].cpu().numpy(), g["phi"])
    if g["n_fv"][0] >= 0:
        assert np.array_equal(r["work"][:, 0].cpu().numpy(), g["n_fv"])


@pytest.mark.parametrize("N", [32, 64, 100, 128, 200, 256, 1024])
def test_forward_fused_within_tolerance(G, N):
    g = golden(f"burgers_forward_N{N}.npz")
    f, pot, _, _ = G.burgers_setup(N, "fused", y=g["y"])
    r = pot.problem().forward(g["u"], want_state=True)
    np.testing.assert_allclose(r["G"].cpu().numpy(), g["G"], rtol=RTOL, atol=1e-13)
    np.testing.assert_allclose(r["phi"].cpu().numpy(), g["phi"], rtol=RTOL)
    np.testing.assert_allclose(r["state"].cpu().numpy(), g["end_state"], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("N", [33, 64, 128, 224, 256, 512, 1024])
def test_forward_fused_positive_and_sign_changing_states(G, N):
    """FUSED runs a select-free time loop when the initial data are positive everywhere and the general
    (upwind-select) loop otherwise (burgers.cuh, flux_fused<.., POS>); both must agree with the
    reference-order solver to the north-star tolerance, on padded and unpadded layouts and for every
    cells-per-lane instantiation of the rotated time loop."""
    P = B.BurgersProblem(N)
    pm = P.prior_mean
    params = np.array([
        [0.025, 0.225, -0.02],     # left 1.025 / right 0.225: positive everywhere
        [1.5, 0.5, 0.3],           # left 2.5 / right 0.5: positive, strong shock
        [0.025, -0.025, -0.02],    # the reference's truth: right state negative (general loop)
        [-0.4, -0.3, 0.1],         # left 0.6 / right -0.3
        [-1.5, 0.4, -0.2],         # left -0.5 / right 0.4: rarefaction through u = 0
        [0.1, 1e-12, 0.0],         # right state barely positive
        [0.1, 0.0, 0.0],           # right state exactly zero (not > 0: general loop)
    ])
    u = params - pm
    fe, pe, _, y = G.burgers_setup(N, "exact")
    ff, pf, _, _ = G.burgers_setup(N, "fused", y=y)
    re_ = pe.problem().forward(u, want_state=True)
    rf = pf.problem().forward(u, want_state=True)
    for i in range(len(u)):
        assert np.array_equal(re_["state"][i].cpu().numpy(), P.end_state(pm + u[i])), (N, i)
    np.testing.assert_array_equal(rf["work"].cpu().numpy()[:, 0], re_["work"].cpu().numpy()[:, 0])
    np.testing.assert_allclose(rf["state"].cpu().numpy(), re_["state"].cpu().numpy(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(rf["G"].cpu().numpy(), re_["G"].cpu().numpy(), rtol=RTOL, atol=1e-13)
    np.testing.assert_allclose(rf["phi"].cpu().numpy(), re_["phi"].cpu().numpy(), rtol=RTOL)


@pytest.mark.parametrize("N", [16, 33, 48, 64, 96, 224, 255, 512])
def test_forward_random_parameters_vs_oracle(G, N):
    """Grids the fixtures do not cover (padded layouts, every CPL instantiation), random u drawn
    from the prior, including shocks starting next to the boundary."""
    rng = np.random.default_rng(N)
    n = 24 if N <= 256 else 6
    u = 0.25 * rng.standard_normal((n, 3))
    u[0] = [0.3, -0.2, 1.49]       # jump right at the right boundary: ghost/IC edge case
    u[1] = [0.3, -0.2, -0.49]      # jump at the left boundary: the left ghost is faster than the
    #                                interior-only CFL allows (rusanov.py:102-109) -> the scheme blows up
    #                                and needs ~100x more steps; lift the engine's safety cap to follow it
    P = B.BurgersProblem(N)
    f, pot, _, y = G.burgers_setup(N, "exact", max_fv_steps=10 ** 6)
    assert np.array_equal(y, P.G_params(G.TRUTH))
    opot = O.Potential(P, y, G.NOISE_COV)
    r = pot.problem().forward(u, want_state=True)
    Gd, phid, st, w = (r[k].cpu().numpy() for k in ("G", "phi", "state", "work"))
    for i in range(n):
        end = P.end_state(P.prior_mean + u[i])
        assert np.array_equal(st[i], end), (N, i)
        assert w[i, 0] == P.last_n_fv
        assert np.array_equal(Gd[i], P.G(u[i]))
        assert phid[i] == opot(u[i])


@pytest.mark.parametrize("N", [33, 64, 128, 256])
def test_fused_on_boundary_ghost_inputs_with_the_cap_lifted(G, N):
    """FUSED numerics on the inputs where the reference's interior-only CFL (rusanov.py:102-109) lets a
    ghost cell sampled from the initial condition (rusanov.py:32) overshoot in the FIRST time step:
    a jump between the left ghost centre and the first cell centre (u = [0.3, -0.2, -0.49] at 64 cells) gives an
    all-positive initial condition (ghost 2.8, interior 0.05) and a sign-changing state after step 1 (min u ~ -4e3).  The select-free positive loop may only be
    entered on the state AFTER the peeled first step (burgers.cuh: state_positive); with the safety cap
    lifted the FUSED solve must follow the reference through the blow-up: same FV step count, G and Phi
    within the north-star tolerance."""
    rng = np.random.default_rng(100 + N)
    P = B.BurgersProblem(N)
    dx = 2.0 / N
    left_gap = (-1 - 0.25 * dx) - P.prior_mean[2]     # jump between the left ghost centre and the first cell centre
    right_gap = (1 + 0.25 * dx) - P.prior_mean[2]     # ... between the last cell centre and the right ghost centre
    u = np.concatenate([[[0.3, -0.2, left_gap], [0.3, -0.2, right_gap], [0.3, 0.2, left_gap], [-0.2, -0.3, left_gap]],
                        np.column_stack([0.25 * rng.standard_normal(8), 0.25 * rng.standard_normal(8),
                                         rng.choice([-0.5, 1.5], 8) + 0.02 * rng.standard_normal(8)])])
    fe, pe, _, y = G.burgers_setup(N, "exact", max_fv_steps=10 ** 7)
    ff, pf, _, _ = G.burgers_setup(N, "fused", y=y, max_fv_steps=10 ** 7)
    opot = O.Potential(P, y, G.NOISE_COV)
    re_ = pe.problem().forward(u, want_state=True)
    rf = pf.problem().forward(u, want_state=True)
    we, wf = re_["work"][:, 0].cpu().numpy(), rf["work"][:, 0].cpu().numpy()
    Ge, Gf, phe, phf = (t.cpu().numpy() for t in (re_["G"], rf["G"], re_["phi"], rf["phi"]))
    assert we.max() > 20 * N                                   # at least one blow-up solve in the batch
    for i in (0, 3):                                           # EXACT is the reference bit for bit, also here
        assert np.array_equal(Ge[i], P.G(u[i])) and we[i] == P.last_n_fv and phe[i] == opot(u[i])
    assert np.array_equal(wf, we)                              # identical step counts
    np.testing.assert_allclose(Gf, Ge, rtol=RTOL, atol=1e-13)
    np.testing.assert_allclose(phf, phe, rtol=RTOL)


@pytest.mark.parametrize("N", [64, 100, 256, 1024, 2048])
def test_monotone_cfl_shortcut_is_bit_identical(G, N):
    """FUSED numerics take max|u| of a state that is monotone in x from its two end cells (burgers.cuh,
    time_loop_mono; the scheme preserves monotonicity, |u| of a monotone profile peaks at an end).  With the
    shortcut switched off (IPMCMC_BURGERS_NO_MONOTONE_SHORTCUT) every solve reduces over all cells: G, Phi, the
    end state and the FV step count must be bit-identical over prior draws incl. rarefactions, sign changes and
    jumps at / outside both boundaries (where the first step breaks monotonicity and the general loop takes over)."""
    import ip_mcmc_b200 as M
    rng = np.random.default_rng(N)
    n = 2048 if N <= 256 else 256
    u = 0.25 * rng.standard_normal((n, 3))
    u[: n // 4, 2] = rng.uniform(-0.55, 1.55, n // 4)
    u[0] = [0.3, -0.2, (-1 - 0.5 / N) + 0.5]         # jump between the left ghost and the first cell centre: blow-up
    a = M.BurgersFVM(N=N, numerics="fused").batch(u, want_state=True)
    b = M.BurgersFVM(N=N, numerics="fused", monotone_shortcut=False).batch(u, want_state=True)
    for k in ("G", "phi", "state", "work"):
        assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), k
    assert a["work"][:, 0].max().item() == 8 * N + 256          # some blow-up solves hit the cap in both


@pytest.mark.parametrize("N", [64, 100, 256, 1000, 1024])
def test_exact_positive_monotone_shortcut_is_bit_identical(G, N):
    """EXACT numerics (the API default) run positive states that are monotone in x through a loop that takes max|u|
    from the upstream end cell and the larger |h| of two neighbours from the direction of the profile, guarded by
    the signs of every difference, and divides without the compiler's slow-path branch (burgers.cuh,
    time_loop_exact_mono).  With the shortcut switched off every solve runs the general code: G, Phi, the end state
    and the FV step count must be the same bits (the golden fixtures pin both to the reference)."""
    import ip_mcmc_b200 as M
    rng = np.random.default_rng(N + 1)
    n = 1024 if N <= 256 else 128
    u = 0.25 * rng.standard_normal((n, 3))
    u[: n // 4, 2] = rng.uniform(-0.55, 1.55, n // 4)
    u[n // 4: n // 2, 0] = rng.uniform(-2.4, -1.0, n // 4)  # left state below the right one: non-decreasing profiles
    u[0] = [0.3, -0.2, (-1 - 0.5 / N) + 0.5]         # jump between the left ghost and the first cell centre: blow-up
    u[1] = [-1.0, 0.25, 0.0]                          # constant state 1.5 (both directions hold)
    a = M.BurgersFVM(N=N, numerics="exact").batch(u, want_state=True)
    b = M.BurgersFVM(N=N, numerics="exact", monotone_shortcut=False).batch(u, want_state=True)
    for k in ("G", "phi", "state", "work"):
        assert np.array_equal(a[k].cpu().numpy(), b[k].cpu().numpy(), equal_nan=True), k


def test_branch_free_division_is_ieee(G):
    """dt = (dx/2) / max|u| of the EXACT positive-monotone loop: the branch-free sequence against the compiler's
    division, bit for bit, over 4M denominators (log-uniform over 12 decades, neighbours of powers of two, ties)."""
    from ip_mcmc_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(7)
    b = np.concatenate([10.0 ** rng.uniform(-6, 6, 1 << 22),
                        np.nextafter(2.0 ** np.arange(-20, 21), np.inf), np.nextafter(2.0 ** np.arange(-20, 21), 0),
                        2.0 ** np.arange(-20.0, 21.0), [3.0, 1.0 / 3.0, 2.525, 0.225, 1e-99, 1e99]])
    bt = G.cuda(b)
    for a in (1.0 / 64, 1.0 / 100, 1.0 / 256, 1.0 / 1000, 1.0 / 1024, 0.1):
        qf, qi = torch.empty_like(bt), torch.empty_like(bt)
        _lib.check(lib.ipmcmc_div_probe(b.size, a, bt.data_ptr(), qf.data_ptr(), qi.data_ptr(), None))
        assert torch.equal(qf, qi), a
        assert np.array_equal(qi.cpu().numpy(), a / b)          # and both are the host's IEEE quotient


def test_callable_interfaces_match_reference_semantics(G):
    """observation_operator(u) -> ndarray[q]; potential(u) -> float (potential.py:53-54)."""
    g = golden("burgers_forward_N64.npz")
    f, pot, _, _ = G.burgers_setup(64, "exact", y=g["y"])
    for i, u in enumerate(g["u"]):
        out = f(u)
        assert isinstance(out, np.ndarray) and out.shape == (5,) and np.array_equal(out, g["G"][i])
        assert pot(u) == g["phi"][i]
        assert pot.exp_minus_potential(u) == np.exp(-g["phi"][i])


def test_step_cap_and_nonfinite_are_reported(G):
    import ip_mcmc_b200 as M
    f = M.BurgersFVM(N=64, max_fv_steps=7)
    r = f.batch(np.zeros((3, 3)))
    assert r["work"][:, 0].tolist() == [7, 7, 7]
    pot = M.EvolutionPotential(f, np.zeros(5), M.GaussianDistribution(np.zeros(5), np.identity(5)))
    assert torch.isnan(pot.batch(np.zeros((2, 3)))["phi"]).all()      # capped solve -> non-finite Phi -> reject
    # an all-zero initial state gives dt = inf and a NaN state, as in the reference (0.5*dx/0)
    f = M.BurgersFVM(N=64)
    r = f.batch(np.array([[-1.0 - 1.5, -0.25, 0.0]]))     # left = 1 + p0 = 0, right = 0
    assert r["work"][0, 0].item() == 1 and torch.isnan(r["G"]).all()


def test_dense_noise_covariance(G):
    """Non-diagonal noise covariance exercises the dense whitening path (scipy eigh factor)."""
    import ip_mcmc_b200 as M
    rng = np.random.default_rng(0)
    A = rng.standard_normal((5, 5))
    cov = 0.01 * (A @ A.T + 5 * np.identity(5))
    g = golden("burgers_forward_N64.npz")
    f = M.BurgersFVM(N=64)
    pot = M.EvolutionPotential(f, g["y"], M.GaussianDistribution(np.zeros(5), cov))
    P = B.BurgersProblem(64)
    opot = O.Potential(P, g["y"], cov)
    phi = pot.batch(g["u"])["phi"].cpu().numpy()
    np.testing.assert_allclose(phi, [opot(u) for u in g["u"]], rtol=1e-12)


def test_full_size_properties(G):
    """BASELINE configs at full size (1024 x 256 and 8192 x 1024 cells): size-independent
    properties -- identical parameters give identical results on every chain (determinism across
    warps/SMs), G of the truth reproduces the data (Phi = the normalisation constant), and the FV
    step count follows ~max|w|*N."""
    for N, n in ((256, 1024), (1024, 8192)):
        f, pot, _, y = G.burgers_setup(N, "exact")
        u = np.tile(G.TRUTH - G.PRIOR_MEAN, (n, 1))
        r = pot.batch(u)
        Gd, phi, w = r["G"].cpu().numpy(), r["phi"].cpu().numpy(), r["work"].cpu().numpy()
        assert np.all(Gd == Gd[0])
        np.testing.assert_allclose(Gd[0], y, rtol=1e-10, atol=1e-12)   # mean + (u* - mean) rounds u* in the last bit
        const = 0.5 * (5 * np.log(2 * np.pi) + np.sum(np.log(np.full(5, 0.05 ** 2))))
        np.testing.assert_allclose(phi, const, rtol=1e-12)
        assert np.all(w[:, 0] == w[0, 0]) and abs(w[0, 0] - 1.027 * N) < 0.02 * N


@pytest.mark.parametrize("N", [2048, 4096])
def test_team_solver_large_grids_vs_oracle(G, N):
    """Grids above 1024 cells run on 2 / 4 warps per chain (burgers_team.cuh): EXACT numerics stay
    bit-identical to the oracle, FUSED within 1e-10; a short chain replays the oracle's decisions."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    rng = np.random.default_rng(N)
    u = np.vstack([G.TRUTH - G.PRIOR_MEAN, 0.25 * rng.standard_normal((2, 3))])
    P = B.BurgersProblem(N)
    f, pot, prior, y = G.burgers_setup(N, "exact")
    assert np.array_equal(y, P.G_params(G.TRUTH))
    opot = O.Potential(P, y, G.NOISE_COV)
    r = pot.problem().forward(u, want_state=True)
    ref_phi = []
    for i in range(len(u)):
        end = P.end_state(P.prior_mean + u[i])
        assert np.array_equal(r["state"][i].cpu().numpy(), end), (N, i)
        assert r["work"][i, 0].item() == P.last_n_fv
        assert np.array_equal(r["G"][i].cpu().numpy(), P.G(u[i]))
        ref_phi.append(opot(u[i]))
        assert r["phi"][i].item() == ref_phi[-1]
    ff, fpot, _, _ = G.burgers_setup(N, "fused", y=y)
    rf = fpot.problem().forward(u)
    np.testing.assert_allclose(rf["phi"].cpu().numpy(), ref_phi, rtol=RTOL)
    np.testing.assert_allclose(rf["G"].cpu().numpy(), r["G"].cpu().numpy(), rtol=RTOL, atol=1e-13)
    # chain replay (pCN beta = 0.25) against the oracle with the same injected noise
    n = 4
    z = 0.25 * rng.standard_normal((n, 3))
    U = rng.random(n)
    start = G.TRUTH - G.PRIOR_MEAN
    ref = O.run_chain(opot, start, z, U, O.PCN, O.PCN, 0.25)
    spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - 0.25 ** 2), coef_w=0.25)
    states, slog, vlog, ch = G.run_injected(pot, spec, start, z, U, n_copies=3)
    for c in range(3):
        assert np.array_equal(states[c], ref["u"]) and np.array_equal(slog[c, :, 0], ref["phi_v"])
    assert ch.counters[:, 1].tolist() == [ref["accepts"]] * 3


@pytest.mark.parametrize("N,m", [(64, 4), (128, 8)])
def test_kl_spectral_extension(G, N, m):
    """North-star item (1): proposals xi from a truncated KL (diagonal, power-law) prior and an
    initial condition carrying the KL modes.  Forward parity against the fixture produced with the
    reference's solver; a pCN chain with d = 3 + m replays the oracle's decisions bit for bit."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    g = golden(f"burgers_kl_N{N}_m{m}.npz")
    f = M.BurgersFVM(N=N, kl_modes=m)
    assert np.array_equal(f.kl_basis, g["basis"]) and f.n_params == 3 + m
    noise = M.GaussianDistribution(np.zeros(5), G.NOISE_COV)
    pot = M.EvolutionPotential(f, g["y"], noise)
    r = pot.problem().forward(g["u"], want_state=True)
    assert np.array_equal(r["state"].cpu().numpy(), g["end_state"])
    assert np.array_equal(r["G"].cpu().numpy(), g["G"]) and np.array_equal(r["phi"].cpu().numpy(), g["phi"])
    assert np.array_equal(f.at_parameters(g["truth"]), g["y"])
    ff = M.BurgersFVM(N=N, kl_modes=m, numerics="fused")
    rf = M.EvolutionPotential(ff, g["y"], noise).problem().forward(g["u"])
    np.testing.assert_allclose(rf["phi"].cpu().numpy(), g["phi"], rtol=RTOL)
    # chain: prior = diag(0.25^2 x3, lambda_k) -> diagonal sample factor sqrt(lambda)
    lam = np.concatenate([np.full(3, 0.25 ** 2), M.BurgersFVM.kl_prior_variances(m)])
    prior = M.GaussianDistribution(f.prior_means, np.diag(lam))
    beta, n = 0.2, 25
    rng = np.random.default_rng(m)
    w = rng.standard_normal((n, 3 + m)) * np.sqrt(lam)
    U = rng.random(n)
    P = B.BurgersProblem(N, kl_basis=g["basis"])
    ref = O.run_chain(O.Potential(P, g["y"], G.NOISE_COV), np.zeros(3 + m), w, U, O.PCN, O.PCN, beta)
    spec = M.SamplerSpec(3 + m, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta)
    states, slog, vlog, ch = G.run_injected(pot, spec, np.zeros(3 + m), w, U, n_copies=2)
    assert np.array_equal(states[0], ref["u"]) and np.array_equal(states[1], ref["u"])
    assert np.array_equal(slog[0, :, 0], ref["phi_v"]) and ref["accepts"] > 0
    # free-running through the public API: Philox z scaled by sqrt(lambda) on the device
    s = M.MCMCSampler(M.ConstSteppCNProposer(beta, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(3))
    out = s.run(np.zeros(3 + m), 200, 0, 1, n_chains=64)
    assert out.shape == (64, 200, 3 + m) and 0.02 < s.accepter.ratio() < 0.95
    spec2, _, _ = s._compile(1, 0, 1, None)
    assert spec2.factor_kind == 1 and np.allclose(np.abs(spec2.factor), np.sqrt(lam))
    # the high modes are weakly informed: their posterior spread stays within the prior's
    post_sd = out[:, 100:, 3:].reshape(-1, m).std(0)
    assert np.all(post_sd < 1.5 * np.sqrt(lam[3:]))


@pytest.mark.parametrize("N,m,numerics", [(128, 61, "exact"), (100, 125, "exact"), (256, 61, "fused"),
                                            (64, 30, "exact"), (64, 30, "fused")])   # d = 33: lane 0 holds u_0 and u_32
def test_kl_prior_beyond_one_warp_of_parameters(G, N, m, numerics):
    """The wide path (32 < d <= 256: parameter vector, proposal and absolute parameters in shared memory;
    include/ipmcmc.h IPMCMC_MAX_DIM_WIDE): a truncated KL prior with m = 30 / 61 / 125 modes.  Forward solves against
    the oracle (whose KL initial condition is pinned to the reference's solver by burgers_kl_*.npz), a pCN and a
    box-constrained RW chain replayed with injected noise (every decision), and free-running chains against the
    oracle driven by the engine's own Philox noise; on-device moments against the recorded trace."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    from oracle import philox_np as Ph
    d = 3 + m
    f = M.BurgersFVM(N=N, kl_modes=m, numerics=numerics)
    P = B.BurgersProblem(N, kl_basis=f.kl_basis)
    rng = np.random.default_rng(m)
    lam = np.concatenate([np.full(3, 0.25 ** 2), M.BurgersFVM.kl_prior_variances(m, scale=0.05)])
    truth = np.concatenate([G.TRUTH, 0.3 * np.sqrt(lam[3:]) * rng.standard_normal(m)])
    y = P.G_params(truth)
    tol = dict(rtol=0, atol=0) if numerics == "exact" else dict(rtol=RTOL, atol=1e-13)
    np.testing.assert_allclose(f.at_parameters(truth), y, **tol)
    noise = M.GaussianDistribution(np.zeros(5), G.NOISE_COV)
    pot = M.EvolutionPotential(f, y, noise)
    opot = O.Potential(P, y, G.NOISE_COV)
    # forward
    u = rng.standard_normal((9, d)) * np.sqrt(lam) * 0.5
    r = pot.problem().forward(u, want_state=True)
    for i in range(9):
        np.testing.assert_allclose(r["G"][i].cpu().numpy(), P.G(u[i]), **tol)
        assert r["work"][i, 0].item() == P.last_n_fv
        np.testing.assert_allclose(r["phi"][i].item(), opot(u[i]), rtol=0 if numerics == "exact" else RTOL)
    # injected-noise replays: pCN, and RW with a box on the shock position
    prior = M.GaussianDistribution(f.prior_means, np.diag(lam))
    n, beta, delta = 20, 0.2, 0.02
    w = rng.standard_normal((n, d)) * np.sqrt(lam)
    U = rng.random(n)
    ref = O.run_chain(opot, np.zeros(d), w, U, O.PCN, O.PCN, beta)
    spec = M.SamplerSpec(d, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta)
    states, slog, vlog, ch = G.run_injected(pot, spec, np.zeros(d), w, U, n_copies=5)
    assert ch.sched is None                                     # static map on the wide path
    for c in (0, 4):
        assert np.array_equal(states[c], ref["u"]) and np.array_equal(vlog[c], ref["v"])
        np.testing.assert_allclose(slog[c, :, 0], ref["phi_v"], rtol=0 if numerics == "exact" else RTOL)
    assert ref["accepts"] > 0 and ch.counters[:, 1].tolist() == [ref["accepts"]] * 5
    lo, hi = -0.62, -0.38
    box = M.BoxConstraint(np.r_[-np.inf, -np.inf, lo, np.full(m, -np.inf)], np.r_[np.inf, np.inf, hi, np.full(m, np.inf)],
                          shift=np.r_[0, 0, -0.5, np.zeros(m)])
    refc = O.run_chain(opot, np.zeros(d), w, U, O.RW, O.RW, delta, prior_cov=np.diag(lam),
                       constraint=lambda v: lo < v[2] - 0.5 < hi, uniforms_by_step=True)
    specc = M.SamplerSpec(d, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * delta), prior_chol=prior.L,
                          constraint=box)
    states, slog, vlog, ch = G.run_injected(pot, specc, np.zeros(d), w, U, n_copies=2)
    assert np.array_equal(states[1], refc["u"])
    valid = ~np.isnan(refc["a"])
    assert ch.counters[1, 5].item() == (~valid).sum() and (~valid).sum() > 0
    np.testing.assert_allclose(slog[1, valid, 1], refc["a"][valid], rtol=1e-12 if numerics == "exact" else 1e-6, atol=1e-300)
    # free-running through the public API, against the oracle with the engine's Philox noise
    s = M.MCMCSampler(M.ConstSteppCNProposer(beta, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(3))
    out = s.run(np.zeros(d), 60, 0, 1, n_chains=37)
    assert out.shape == (37, 60, d)
    for c in (0, 36):
        z, Uc = Ph.chain_noise(s.last_run["seed"], c, 0, 60, d)
        refp = O.run_chain(opot, np.zeros(d), z * np.sqrt(lam), Uc, O.PCN, O.PCN, beta)
        np.testing.assert_allclose(out[c], refp["u"], rtol=1e-12 if numerics == "exact" else 1e-9, atol=1e-14)
    flat = out.reshape(-1, d)
    np.testing.assert_allclose(s.last_run["pooled_mean"], flat.mean(0), rtol=1e-9, atol=1e-14)
    np.testing.assert_allclose(s.last_run["pooled_var"], flat.var(0, ddof=1), rtol=1e-8)
    # the host entry point takes the same path
    h = M.MCMCSampler(M.ConstSteppCNProposer(beta, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(3))
    assert np.array_equal(h.run_host(np.zeros(d), 60, 0, 1, n_chains=37), out)
