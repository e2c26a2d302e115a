"""GPU parity of the fused Metropolis kernel: the reference's own chains (recorded with a noise
tape, tests/golden/chain_*.npz) replayed with injected noise must be reproduced state by state."""
import numpy as np
import pytest
import torch

from conftest import golden
from oracle import burgers_np as B
from oracle import mcmc_np as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def G():
    import gpu_common
    return gpu_common


def _spec(kind, g, prior, **kw):
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    if kind == "pcn":
        beta = float(g["beta"])
        return M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - beta ** 2), coef_w=beta, **kw)
    delta = float(g["delta"])
    return M.SamplerSpec(3, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * delta),
                         prior_chol=prior.L, **kw)


NUMERICS = ["exact", "fused"]


def _check_phi(numerics, got, want):
    """EXACT: bit-identical; FUSED (the numerics bench.py measures): north-star tolerance 1e-10 relative."""
    if numerics == "exact":
        assert np.array_equal(got, want)
    else:
        np.testing.assert_allclose(got, want, rtol=1e-10)


@pytest.mark.parametrize("numerics", NUMERICS)
@pytest.mark.parametrize("name,kind", [("chain_burgers_pcn_N64.npz", "pcn"), ("chain_burgers_pcn_N128.npz", "pcn"),
                                       ("chain_burgers_rw_N64.npz", "rw"),
                                       ("chain_burgers_pcn_N256.npz", "pcn"),              # the bench grid, from u_0 = 0
                                       ("chain_burgers_pcn_N256_continued.npz", "pcn")])   # ... and 150 steps further on
def test_replay_reference_chain(G, name, kind, numerics):
    """The reference's own chain (MCMCSampler.run with a noise tape, oracle/make_golden.py) replayed with
    the tape injected: every proposal, every accept decision (hence every state) and every Phi(v)."""
    g = golden(name)
    f, pot, prior, _ = G.burgers_setup(int(g["N"]), numerics)
    states, slog, vlog, ch = G.run_injected(pot, _spec(kind, g, prior), g["u0"], g["normals"], g["uniforms"], n_copies=3)
    acc_ref = np.all(g["samples"] == g["v"], axis=1)
    for c in range(3):
        assert np.array_equal(states[c], g["samples"])                 # all accept decisions
        assert np.array_equal(vlog[c], g["v"])
        _check_phi(numerics, slog[c, :, 0], g["phi_v"])
        assert np.array_equal(slog[c, :, 2].astype(bool), acc_ref) and int(slog[c, :, 2].sum()) == int(g["accepts"])
    cnt = ch.counters.cpu().numpy()
    assert np.all(cnt[:, 0] == int(g["calls"])) and np.all(cnt[:, 1] == int(g["accepts"]))
    assert np.all(cnt[:, 3] == len(g["normals"]) + 1)      # one solve per step + Phi(u_0)
    # accept probabilities vs the oracle's exp (device exp is <= 1 ulp from libm)
    if kind == "pcn":
        a_ref = np.exp(g["phi_u"] - g["phi_v"])
        np.testing.assert_allclose(slog[0, :, 1], a_ref, rtol=1e-14 if numerics == "exact" else 1e-6, atol=1e-300)
        # no decision of this tape is borderline at the FUSED tolerance: |a - U| >> 1e-10 * a * Phi
        assert np.min(np.abs(a_ref - g["uniforms"]) / np.maximum(a_ref, 1e-300)) > 1e-6


def test_recompute_phi_u_is_bit_equivalent_for_burgers(G):
    """The reference evaluates Phi(u) again every step (accepter.py:121-122); for a deterministic
    G caching is bit-equivalent -- checked by running the kernel both ways."""
    g = golden("chain_burgers_pcn_N64.npz")
    f, pot, prior, _ = G.burgers_setup(64)
    s1, l1, _, c1 = G.run_injected(pot, _spec("pcn", g, prior), g["u0"], g["normals"], g["uniforms"])
    s2, l2, _, c2 = G.run_injected(pot, _spec("pcn", g, prior, recompute_phi_u=True), g["u0"], g["normals"], g["uniforms"])
    assert np.array_equal(s1, s2) and np.array_equal(l1[..., :3], l2[..., :3])
    assert c2.counters[0, 3].item() == 2 * len(g["normals"]) + 1   # the reference's 2 solves per step


@pytest.mark.parametrize("numerics", NUMERICS)
def test_replay_varstep_schedule(G, numerics):
    """VarStepStandardRWProposer with the PWLinear schedule (proposer.py:33-56, burgers_beta.py:131-147)."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    g = golden("chain_burgers_varstep_rw_N64.npz")
    f, pot, prior, _ = G.burgers_setup(64, numerics)
    sched = np.stack([np.ones(len(g["schedule"])), np.sqrt(2) * np.sqrt(g["schedule"])], axis=1)
    spec = M.SamplerSpec(3, _lib.PROPOSE_RW, _lib.ACCEPT_RW, schedule=sched, prior_chol=prior.L)
    states, slog, _, ch = G.run_injected(pot, spec, g["u0"], g["normals"], g["uniforms"])
    assert np.array_equal(states[0], g["samples"])
    _check_phi(numerics, slog[0, :, 0], g["phi_v"])
    assert ch.counters[0, 1].item() == int(g["accepts"])


@pytest.mark.parametrize("numerics", NUMERICS)
def test_replay_constrained_chain(G, numerics):
    """ConstrainAccepter: a violated box rejects WITHOUT consuming a uniform (accepter.py:52-55)."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    g = golden("chain_burgers_constrained_rw_N64.npz")
    f, pot, prior, _ = G.burgers_setup(64, numerics)
    lo, hi = float(g["lo"]), float(g["hi"])
    box = M.BoxConstraint([-np.inf, -np.inf, lo], [np.inf, np.inf, hi], shift=[0, 0, -0.5])
    # expand the tape: the reference drew U only on the steps whose proposal satisfied the box
    P = B.BurgersProblem(64)
    opot = O.Potential(P, P.G_params(G.TRUTH), G.NOISE_COV)
    ref = O.run_chain(opot, g["u0"], g["normals"], g["uniforms"], O.RW, O.RW, float(g["delta"]),
                      prior_cov=G.PRIOR_COV, constraint=lambda v: lo < v[2] - 0.5 < hi)
    assert np.array_equal(ref["u"], g["samples"])
    valid = ~np.isnan(ref["a"])
    U = np.full(len(g["normals"]), 0.5)
    U[valid] = g["uniforms"]
    spec = M.SamplerSpec(3, _lib.PROPOSE_RW, _lib.ACCEPT_RW, coef_u=1.0, coef_w=np.sqrt(2 * float(g["delta"])),
                         prior_chol=prior.L, constraint=box)
    states, slog, _, ch = G.run_injected(pot, spec, g["u0"], g["normals"], U)
    assert np.array_equal(states[0], g["samples"])
    cnt = ch.counters[0].cpu().numpy()
    assert cnt[0] == int(g["calls"]) and cnt[1] == int(g["accepts"])
    assert cnt[5] == (~valid).sum() and cnt[3] == valid.sum() + 1   # no solve on constrained steps


def test_sampler_api_step_accounting_and_counters(G):
    """MCMCSampler.run keeps the reference's accounting (sampler.py:12-33, sampler_test.py:8-18):
    max(0, burn_in - interval) + n*interval calls, counter reset when outermost, shapes."""
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(32)
    acc = M.CountedAccepter(M.pCNAccepter(pot))
    s = M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), acc, np.random.default_rng(2))
    out = s.run(np.zeros(3), 27, burn_in=20, sample_interval=10)
    assert out.shape == (27, 3) and acc.calls == 280
    assert 0 < acc.accepts < 280 and acc.ratio() == acc.accepts / 280
    out = s.run(np.zeros(3), 5, 0, 1, n_chains=7)
    assert out.shape == (7, 5, 3) and acc.calls == 35          # reset, then 7 chains x 5 steps
    assert s.last_run["counters"]["work_b"] == 7 * 6
    with pytest.raises(TypeError):
        M.EvolutionPotential(lambda u: u, np.zeros(5), None)     # no CPU fallback for Python G
    with pytest.raises(TypeError):
        M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.ConstrainAccepter(M.pCNAccepter(pot), lambda v: True),
                      np.random.default_rng(0)).run(np.zeros(3), 1, 0, 1)


def test_recording_moments_and_chunked_launches(G):
    """Thinning/burn-in slicing matches the reference definition; on-device Welford moments equal
    the moments of the recorded trace; chunked launches and one launch give identical chains."""
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(32)
    mk = lambda: M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.CountedAccepter(M.pCNAccepter(pot)),
                               np.random.default_rng(5))
    s_all = mk()
    every = s_all.run(np.zeros(3), 130, 0, 1, n_chains=16)
    s_thin = mk()
    thin = s_thin.run(np.zeros(3), 12, burn_in=20, sample_interval=10, n_chains=16)
    assert np.array_equal(thin, O.samples_from_states(every.transpose(1, 0, 2), 12, 20, 10).transpose(1, 0, 2))
    s_chunk = mk()
    chunk = s_chunk.run(np.zeros(3), 12, burn_in=20, sample_interval=10, n_chains=16, steps_per_launch=17)
    assert np.array_equal(chunk, thin) and s_chunk.last_run["launches"] > 3
    lr = s_thin.last_run
    flat = thin.reshape(-1, 3)
    assert lr["pooled_count"] == flat.shape[0]
    np.testing.assert_allclose(lr["pooled_mean"], flat.mean(0), rtol=1e-12)
    np.testing.assert_allclose(lr["pooled_var"], flat.var(0, ddof=1), rtol=1e-10)


def test_results_do_not_depend_on_sharding(G):
    """Philox is keyed by the GLOBAL chain id: 12 chains in one batch == 3 shards of 4."""
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(32)
    mk = lambda: M.MCMCSampler(M.ConstStepStandardRWProposer(0.01, prior), M.StandardRWAccepter(pot, prior),
                               np.random.default_rng(9))
    whole = mk().run(np.zeros(3), 40, 0, 1, n_chains=12)
    parts = [mk().run(np.zeros(3), 40, 0, 1, n_chains=4, chain_offset=4 * r) for r in range(3)]
    assert np.array_equal(whole, np.concatenate(parts, axis=0))
    assert not np.array_equal(whole[0], whole[1])


def test_engine_rng_matches_cpu_statement(G):
    from ip_mcmc_b200 import _lib
    from oracle import philox_np as P
    lib = _lib.load()
    seed = 2 + (5 << 32)
    out = torch.empty((3, 40, 4), dtype=torch.float64, device="cuda")
    _lib.check(lib.ipmcmc_rng_probe(seed, 7, (1 << 33) + 5, 3, 40, 3, out.data_ptr(), None))
    o = out.cpu().numpy()
    for c in range(3):
        z, U = P.chain_noise(seed, 7 + c, (1 << 33) + 5, 40, 3)
        assert np.array_equal(o[c, :, 3], U)                    # integers -> uniforms: bit exact
        np.testing.assert_allclose(o[c, :, :3], z, rtol=0, atol=1e-13)   # log/sqrt/cos: few ulp


def test_free_running_chain_statistics_vs_cpu_oracle(G):
    """Statistical parity (SURVEY.md section 8(d)): acceptance rate and posterior mean of
    free-running device chains vs CPU oracle chains, within Monte Carlo error."""
    import ip_mcmc_b200 as M
    N, beta, n_steps, burn = 32, 0.25, 600, 200
    f, pot, prior, y = G.burgers_setup(N)
    s = M.MCMCSampler(M.ConstSteppCNProposer(beta, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(2))
    dev = s.run(np.zeros(3), n_steps, 0, 1, n_chains=256)
    P = B.BurgersProblem(N)
    opot = O.Potential(P, y, G.NOISE_COV)
    rng = np.random.default_rng(3)
    cpu_states, cpu_acc = [], []
    for c in range(6):
        z = 0.25 * rng.standard_normal((n_steps, 3))
        r = O.run_chain(opot, np.zeros(3), z, rng.random(n_steps), O.PCN, O.PCN, beta)
        cpu_states.append(r["u"][burn:])
        cpu_acc.append(r["accepted"][burn:].mean())
    cpu = np.concatenate(cpu_states)
    dev_post = dev[:, burn:].reshape(-1, 3)
    # device: 256 chains x 400 steps; cpu: 6 x 400.  MCSE dominated by the CPU side.
    ess_cpu = sum(M.stats.ess(st).min() for st in cpu_states)
    mcse = cpu.std(0) / np.sqrt(max(ess_cpu, 4))
    assert np.all(np.abs(dev_post.mean(0) - cpu.mean(0)) < 5 * mcse + 1e-3), (dev_post.mean(0), cpu.mean(0), mcse)
    acc_dev = s.last_run["per_chain_counters"][:, 1].double().mean().item() / n_steps
    assert abs(acc_dev - np.mean(cpu_acc)) < 0.12
    # both samplers have left the prior-mean start in the same direction (towards delta_1 = u*_1)
    assert dev_post.mean(0)[0] < -0.3 and cpu.mean(0)[0] < -0.3


def test_host_buffer_entry_point_matches_device_path(G):
    """ipmcmc_sample_host (host pointers in/out, copies inside; MCMCSampler.run_host) == MCMCSampler.run on
    the same seed -- samples, counters, pooled moments, final states -- and continued from a known Phi(u_0)
    without the extra solve."""
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(32, "fused")
    mk = lambda: M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.CountedAccepter(M.pCNAccepter(pot)), np.random.default_rng(4))
    n_chains, n = 9, 25
    s = mk()
    ref = s.run(np.zeros(3), n, 0, 1, n_chains=n_chains)
    h = mk()
    got = h.run_host(np.zeros(3), n, 0, 1, n_chains=n_chains)
    assert h.last_run["seed"] == s.last_run["seed"]
    assert np.array_equal(got, ref)
    assert np.array_equal(h.last_run["per_chain_counters"], s.last_run["per_chain_counters"].cpu().numpy())
    assert h.accepter.calls == n_chains * n and h.accepter.accepts == s.accepter.accepts
    assert h.last_run["pooled_count"] == n_chains * n
    np.testing.assert_allclose(h.last_run["pooled_mean"], ref.reshape(-1, 3).mean(0), rtol=1e-12)
    np.testing.assert_allclose(h.last_run["pooled_var"], ref.reshape(-1, 3).var(0, ddof=1), rtol=1e-10)
    assert np.array_equal(h.last_run["u"], ref[:, -1]) and np.array_equal(h.last_run["phi"], s.last_run["phi"].cpu().numpy())
    # continuation with a known Phi(u_0): one solve per step, none for u_0; same as the device path
    a, b = mk(), mk()
    ra = a.run(s.last_run["u"], 10, 0, 1, phi_0=s.last_run["phi"])
    rb = b.run_host(h.last_run["u"], 10, 0, 1, phi_0=h.last_run["phi"])
    assert np.array_equal(ra, rb)
    assert a.last_run["counters"]["work_b"] == n_chains * 10 == b.last_run["counters"]["work_b"]
    c = mk()
    rc = c.run(s.last_run["u"], 10, 0, 1)
    assert np.array_equal(rc, ra) and c.last_run["counters"]["work_b"] == n_chains * 11


@pytest.mark.parametrize("N,n_chains,steps_per_launch", [(32, 700, None), (64, 1500, 5), (256, 1024, 7), (100, 333, 3)])
def test_queue_is_pure_scheduling(G, N, n_chains, steps_per_launch, monkeypatch):
    """The dynamic step scheduler (persistent warps + FIFO of ready chains, chain state travelling through L2
    between work items) is pure scheduling: samples, per-chain counters and Welford moments are the same bits
    with the default work items (4 steps for a 262-step launch) and CTA shape in one launch, and with one step
    per item, one warp per SM when the batch is one wave (148 warps serve hundreds of chains, which change warps
    at almost every step) and the launch split (small batch, > 8 n_SM batch, the bench shape, a padded grid)."""
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(N, "fused")
    mk = lambda: M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.CountedAccepter(M.pCNAccepter(pot)),
                               np.random.default_rng(8))
    a, b = mk(), mk()
    out_a = a.run(np.zeros(3), 130, 4, 2, n_chains=n_chains)
    monkeypatch.setenv("IPMCMC_SCHED_CHUNK", "1")
    monkeypatch.setenv("IPMCMC_SCHED_WPC", "1")          # read for one-wave batches (<= 8 n_SM chains) only
    out_b = b.run(np.zeros(3), 130, 4, 2, n_chains=n_chains, steps_per_launch=steps_per_launch)
    ca, cb = a.last_run["chains"], b.last_run["chains"]
    assert ca.sched is not None and cb.sched is not None
    assert np.array_equal(out_a, out_b)
    assert torch.equal(ca.counters, cb.counters) and torch.equal(ca.u, cb.u) and torch.equal(ca.phi, cb.phi)
    assert torch.equal(ca.mom_count, cb.mom_count) and torch.equal(ca.mom_mean, cb.mom_mean) and torch.equal(ca.mom_m2, cb.mom_m2)
    assert a.accepter.calls == b.accepter.calls and a.accepter.accepts == b.accepter.accepts


def test_library_allocates_queue_scratch(G):
    """ipmcmc_run without scheduler scratch (sched_dev = NULL) runs the queue on a stream-ordered allocation of the
    library's: the same bits as with ChainBatch's scratch, over two launches."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import _lib
    f, pot, prior, _ = G.burgers_setup(64, "fused")
    spec = M.SamplerSpec(3, _lib.PROPOSE_PCN, _lib.ACCEPT_PCN, coef_u=np.sqrt(1 - 0.25 ** 2), coef_w=0.25,
                         factor=np.full(3, 0.25), seed=11)
    runs = []
    for own in (True, False):
        ch = M.ChainBatch(pot.problem(), np.zeros(3), n_chains=300)
        assert ch.sched is not None
        if not own:
            ch.sched = None
        traces = [torch.empty((300, 20, 3), dtype=torch.float64, device="cuda") for _ in range(2)]
        for t in traces:
            ch.run(spec, 20, trace=t)
        runs.append((torch.cat(traces, 1), ch))
    (ta, ca), (tb, cb) = runs
    assert torch.equal(ta, tb) and ca.counters[:, 1].sum().item() > 0
    for name in ("u", "phi", "counters", "mom_count", "mom_mean", "mom_m2"):
        assert torch.equal(getattr(ca, name), getattr(cb, name)), name


def test_grid_refinement_study_driver(G):
    """Engine-side half of burgers_wasserstein_grid.py: VarStep RW + box-constrained accepter on
    several grids, 3-D histograms on the device."""
    from ip_mcmc_b200 import studies
    out = studies.grid_refinement_study(grids=(32, 64), n_steps=300, n_chains=32, burn_in=100)
    for N in (32, 64):
        h = out[N]["histogram"]
        assert h.shape == (20, 20, 20) and abs(h.sum() * 0.05 ** 3 - 1) < 1e-9
        assert 0.01 < out[N]["acceptance"] < 0.99


def test_device_histogram_matches_numpy(G):
    """ipmcmc_histogram_accumulate == np.histogramdd (right-open bins, last edge inclusive, outside dropped),
    accumulated over several calls, with values exactly on edges and a padded row stride."""
    from ip_mcmc_b200 import studies
    rng = np.random.default_rng(3)
    iv = np.array([[-0.5, 0.5], [0.0, 2.0], [-1.0, 0.25]])
    x = rng.standard_normal((20000, 3)) * [0.3, 0.8, 0.5] + [0.0, 1.0, -0.4]
    edges = [np.linspace(lo, hi, 21) for lo, hi in iv]
    x[:21, 0] = edges[0]                     # on every edge of dimension 0 (incl. both ends)
    x[21:42, 1] = edges[1]
    x[50] = [0.5, 2.0, 0.25]                 # the upper corner belongs to the last bin
    shift = np.array([0.1, -0.2, 0.05])
    h = studies.DeviceHistogram(iv, bins=20, shift=shift)
    xs = x - shift
    padded = np.concatenate([xs, np.full((len(xs), 2), 99.0)], axis=1)       # stride 5: extra columns ignored
    h.add(G.cuda(padded[:7000]))
    h.add(G.cuda(xs[7000:]))
    ref, _ = np.histogramdd(xs + shift, bins=20, range=iv)
    assert np.array_equal(h.counts.cpu().numpy(), ref.astype(np.int64))
    np.testing.assert_allclose(h.normalised(), ref / ref.sum(), rtol=1e-15)


def test_chain_length_study_streams_the_same_histograms(G):
    """chain_length_study (burgers_wasserstein_chain.py:164-268 on the device): the histograms accumulated launch
    by launch equal np.histogramdd of the same chains recorded in full and split as the script does; and the
    chains themselves equal the CPU oracle run with the engine's own Philox noise (VarStep RW + box constraint)."""
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import studies
    from oracle import philox_np as P
    N, L, si, B_ = 32, 1200, 5, 3
    r = studies.chain_length_study(chain_length=L, n_chains=B_, N=N, sample_interval=si, steps_per_launch=170, seed=7)
    # the same chains recorded in full through the public sampler (same seed, same object graph)
    pm = np.array([1.5, 0.25, -0.5])
    f, pot, prior, _ = G.burgers_setup(N)
    sched = studies.PWLinear(0.05, 0.001, 250)
    box = M.BoxConstraint([-np.inf, -np.inf, -1.0], [np.inf, np.inf, 1.0], shift=[0.0, 0.0, pm[2]])
    counted = M.CountedAccepter(M.StandardRWAccepter(pot, prior))
    s = M.MCMCSampler(M.VarStepStandardRWProposer(sched, prior), M.ConstrainAccepter(counted, box), np.random.default_rng(7))
    full = s.run(np.zeros(3), L, 0, 1, n_chains=B_)                     # [B, L, 3]
    thinned = full[:, ::si] + pm
    chains, rest = [], thinned
    for _ in range(4):                                                  # burgers_wasserstein_chain.py:261-266
        l = rest.shape[1] // 2
        chains.append(rest[:, l + 1:])
        rest = rest[:, :l]
    iv = np.stack([np.min([c.reshape(-1, 3).min(0) for c in chains], axis=0),
                   np.max([c.reshape(-1, 3).max(0) for c in chains], axis=0)], axis=1)
    np.testing.assert_array_equal(r["intervals"], iv)
    for k, c in enumerate(chains):
        ref, _ = np.histogramdd(c.reshape(-1, 3), bins=20, range=iv)
        assert np.array_equal(r["counts"][k], ref.astype(np.int64)), k
        assert r["lengths"][k] == c.shape[1]
    assert r["acceptance"] == pytest.approx(counted.ratio())            # counter inside the constraint
    # ... and chain 1 against the CPU oracle with the engine's noise
    z, U = P.chain_noise(s.last_run["seed"], 1, 0, L, 3)
    Pb = B.BurgersProblem(N)
    opot = O.Potential(Pb, Pb.G_params(G.TRUTH), G.NOISE_COV)
    steps = np.array([sched(i) for i in range(1, L + 1)])
    ref = O.run_chain(opot, np.zeros(3), 0.25 * z, U, O.RW, O.RW, steps, prior_cov=G.PRIOR_COV, varstep=True,
                      constraint=lambda v: -1.0 < v[2] + pm[2] < 1.0, uniforms_by_step=True)
    np.testing.assert_allclose(full[1], ref["u"], rtol=1e-12, atol=1e-14)


def test_chain_length_study_at_the_reference_scale(G):
    """The script's own size (burgers_wasserstein_chain.py:165: 100 000 steps, N = 128, thinning 20) for 64 chains:
    4 x 20^3 counters instead of 64 x 100 000 x 3 samples; every thinned sample of every sub-chain lands in a bin
    (the intervals are the sub-chains' own extrema), longer sub-chains concentrate around the truth's bin."""
    from ip_mcmc_b200 import studies
    r = studies.chain_length_study(chain_length=100000, n_chains=64, steps_per_launch=10000)
    assert r["lengths"] == [2499, 1249, 624, 312]                       # 5000 thinned samples, halved four times
    for k, n in enumerate(r["lengths"]):
        assert int(r["counts"][k].sum()) == 64 * n
        np.testing.assert_allclose(r["histograms"][k].sum(), 1.0, rtol=1e-12)
    assert 0.05 < r["acceptance"] < 0.95 and r["ground_truth_bin"] is not None
    # marginal of delta_1 (axis 0): the posterior mass sits within a few bins of the truth's bin
    gt = r["ground_truth_bin"][0]
    marg = r["histograms"][0].sum(axis=(1, 2))
    assert marg[max(gt - 4, 0):gt + 5].sum() > 0.5


def test_run_into_preallocated_host_buffer(G):
    """`out=`: samples land in a caller-owned (pinned torch or NumPy) host buffer, identical to the
    returned-array path; wrong sizes are refused."""
    import ip_mcmc_b200 as M
    f, pot, prior, _ = G.burgers_setup(64, "fused")
    mk = lambda: M.MCMCSampler(M.ConstSteppCNProposer(0.25, prior), M.CountedAccepter(M.pCNAccepter(pot)),
                               np.random.default_rng(3))
    ref = mk().run(np.zeros(3), 9, 0, 1, n_chains=17)
    pinned = torch.empty((17, 9, 3), dtype=torch.float64).pin_memory()
    got = mk().run(np.zeros(3), 9, 0, 1, n_chains=17, out=pinned)
    assert np.array_equal(got, ref) and np.array_equal(pinned.numpy(), ref)
    arr = np.empty((17, 9, 3))
    got2 = mk().run(np.zeros(3), 9, 0, 1, n_chains=17, out=arr)
    assert np.array_equal(arr, ref) and got2 is not None
    with pytest.raises(ValueError):
        mk().run(np.zeros(3), 9, 0, 1, n_chains=17, out=np.empty((17, 8, 3)))
