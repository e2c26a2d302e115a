#!/usr/bin/env python
"""bench.py -- MCMC chain-steps/s (and ESS/s) of the fused Metropolis kernel on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, NCCL)

A "step" is ONE launch of the fused kernel advancing every chain of the batch by `--mcmc-steps`
Metropolis steps (proposal -> forward solve -> Phi -> accept/reject -> moments; default 1000 / 16 / 128 steps per
launch for the three workloads, see WORKLOADS).  Workloads
(BASELINE.json `configs`):
    burgers_pcn_256   configs[2]: Burgers pCN beta=0.25, 1024 chains x 256 cells per GPU   (default)
    burgers_pcn_1024  configs[3]: Burgers pCN, 8192 chains x 1024 cells per GPU (65536 over 8 GPUs)
    lorenz_rw         configs[1]: Lorenz-96 K=6 J=4 T=20, RW delta=0.125, 4096 chains per GPU
The default run (burgers_pcn_256) also measures the other two as `extra_workloads` (at every N), the same
workload with the EXACT numerics, a COLD START leg (the reference's u_0 = 0, 5000 steps in one launch, no
burn-in: burgers_mcmc.py:129-134) and the C entry point with host buffers (`e2e_c_abi`).
Scaling is weak: the per-GPU batch is fixed, chains are sharded by global chain id, no data-path
collective; one all-reduce of pooled moments/counters at the end (inside the timed region).

`--impl reference` times the CPU restatement of the reference's sampler (oracle/, NumPy; the
reference itself is pure Python + NumPy and cannot travel to the GPU box) on all host cores.

`--dump-outputs DIR` writes what the last timed launch of the main workload returned, as float64 .npy files:
samples (the recorded states, [chains, mcmc_steps, 3]), u and phi (the final state and Phi of every chain),
model_state (Lorenz only: the carried initial condition) and pooled (the all-reduced moments and counters).
The inputs are seeded, so two builds run with the same arguments can be compared array by array.  Above 64 MB
a fixed, seeded subset of the chains is written, with their global ids in chain_index.  With several GPUs,
rank 0 writes its own chains and the global pooled moments.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TRUTH = np.array([0.025, -0.025, -0.02])
PRIOR_MEAN = np.array([1.5, 0.25, -0.5])

# Metropolis steps per launch (= per bench "step").  MCMCSampler.run(n_steps) is ONE launch whatever n_steps is, and the
# reference's chains are 5000+ steps long; a launch ends when its slowest chain ends, and with as many resident warps as
# chains nothing can be rebalanced at the end, so short launches pay the spread of per-chain work once per launch
# (1024 x 256 cells: 200-step launches 70.9 %, 1000-step launches 74.0 % of the DFMA peak, 5000 steps 74.8 %).
# Round 1 and the first half of round 2 timed 200 / 4 / 32 steps per launch; that figure is still reported
# (`short_launch`).
WORKLOADS = {
    "burgers_pcn_256": dict(model="burgers", N=256, chains=1024, mcmc_steps=1000, beta=0.25),
    "burgers_pcn_1024": dict(model="burgers", N=1024, chains=8192, mcmc_steps=16, beta=0.25),
    "lorenz_rw": dict(model="lorenz", chains=4096, mcmc_steps=128, delta=0.125, T=20.0),
}
SHORT_LAUNCH_STEPS = 200
DUMP_LIMIT_BYTES = 64 * 10 ** 6


# ------------------------------------------------------------------------------------------------
# CPU side (oracle port): used by the cpu_baseline leg and by --impl reference
# ------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """Advance ONE chain by n_steps with the NumPy restatement of the reference sampler."""
    wl, seed, n_steps, u_start = args
    from oracle import burgers_np as B, mcmc_np as O, lorenz_np as L
    rng = np.random.default_rng(seed)
    if wl["model"] == "burgers":
        P = B.BurgersProblem(wl["N"])
        y = P.G_params(TRUTH)
        pot = O.Potential(P, y, 0.05 ** 2 * np.identity(5))
        z = 0.25 * rng.standard_normal((n_steps, 3))
        t0 = time.perf_counter()
        # the reference evaluates Phi(u) and Phi(v) every step (accepter.py:121-122)
        r = O.run_chain(pot, u_start, z, rng.random(n_steps), O.PCN, O.PCN, wl["beta"], recompute_phi_u=True)
        return time.perf_counter() - t0, n_steps, r["accepts"], P.total_n_fv
    g = np.load(os.path.join(ROOT, "tests", "golden", "lorenz_problem_K6_J4.npz"))
    op = L.LorenzProblem(6, 4, wl["T"], 1, g["prior_means"], g["IC"])
    pot = O.Potential(op, g["y"], 0.25 * np.diag(g["var"]))
    z = rng.standard_normal((n_steps, 3)) * np.sqrt([10., 1, 10])
    t0 = time.perf_counter()
    r = O.run_chain(pot, g["u0"], z, rng.random(n_steps), O.RW, O.RW, wl["delta"],
                    prior_cov=np.diag([10., 1, 10]), recompute_phi_u=True)
    return time.perf_counter() - t0, n_steps, r["accepts"], op.n_accepted + op.n_rejected


def cpu_sample(wl, n_steps, n_workers, u_start):
    """n_workers independent chains x n_steps on n_workers processes. Returns chain-steps/s."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(n_workers) as pool:
        res = pool.map(_cpu_worker, [(wl, 1000 + i, n_steps, u_start) for i in range(n_workers)])
    wall = time.perf_counter() - t0
    busy = max(r[0] for r in res)
    steps = sum(r[1] for r in res)
    return steps / busy, busy, wall, res


def cpu_acceptance(res):
    return sum(r[2] for r in res) / max(1, sum(r[1] for r in res))


def cpu_sample_c(wl, n_steps, n_threads, u_start):
    """The same chains through the plain-C restatement (oracle/oracle_c.c; 2 forward solves per step like the
    reference), one chain per host thread.  A much faster CPU figure than the NumPy port, reported beside it."""
    from oracle import c_oracle as CO, burgers_np as B
    rng = np.random.default_rng(1000)
    U = rng.random((n_threads, n_steps))
    if wl["model"] == "burgers":
        P = CO.BurgersC(wl["N"], y=B.BurgersProblem(wl["N"]).G_params(TRUTH), noise_cov=0.05 ** 2 * np.identity(5))
        z = 0.25 * rng.standard_normal((n_threads, n_steps, 3))
        t0 = time.perf_counter()
        r = P.run_chains(u_start, z, U, CO.PCN, CO.PCN, wl["beta"], recompute_phi_u=True, n_threads=n_threads)
    else:
        g = np.load(os.path.join(ROOT, "tests", "golden", "lorenz_problem_K6_J4.npz"))
        L = CO.LorenzC(6, 4, wl["T"], 1.0, g["prior_means"], y=g["y"], noise_cov=0.25 * np.diag(g["var"]))
        z = rng.standard_normal((n_threads, n_steps, 3)) * np.sqrt([10., 1, 10])
        t0 = time.perf_counter()
        r = L.run_chains(g["u0"], g["IC"], z, U, CO.RW, CO.RW, wl["delta"], prior_cov=np.diag([10., 1, 10]), n_threads=n_threads)
    dt = time.perf_counter() - t0
    return n_threads * n_steps / dt, dt, float(r["accepted"].mean())


def cpu_baselines(wl, cores):
    """cpu_baseline (NumPy port, the contract's key) and cpu_baseline_c (plain-C port) of one workload."""
    n = cpu_steps_for(wl)
    v, busy, wall, res = cpu_sample(wl, n, cores, posterior_start(wl))
    out = dict(cpu_baseline=dict(value=v, unit="chain-steps/s", cores=cores, kind="port", acceptance=cpu_acceptance(res),
                                 sample="%d processes x %d chain-steps of the same workload, NumPy restatement of the "
                                        "reference sampler (2 forward solves per step), %.1f s" % (cores, n, busy)))
    try:
        n_c = {"burgers": 1500 if wl.get("N", 0) <= 256 else 40, "lorenz": 60}[wl["model"]]
        vc, dtc, acc_c = cpu_sample_c(wl, n_c, cores, posterior_start(wl))
        out["cpu_baseline_c"] = dict(value=vc, unit="chain-steps/s", cores=cores, kind="port (plain C, oracle/oracle_c.c)",
                                     acceptance=acc_c, sample="%d threads x %d chain-steps, 2 forward solves per step, %.1f s"
                                                              % (cores, n_c, dtc))
    except Exception as e:      # the C oracle is test infrastructure: never let it break the bench line
        out["cpu_baseline_c"] = dict(unavailable=str(e)[:200])
    return out


def cpu_steps_for(wl):
    # bounded sample per process (16 of them on the box's 16 cores): ~13 s at N = 256 (~70 chain-steps/s/core),
    # ~3 s at N = 1024 (~13 /s/core), ~5 s Lorenz (~1.2 /s/core)
    return {"burgers": 900 if wl.get("N", 0) <= 256 else 40, "lorenz": 6}[wl["model"]]


def posterior_start(wl):
    """A state near the posterior, so the CPU sample does the same kind of work as the warmed-up
    GPU chains (solves from the prior mean cost 2.4x more FV steps, SURVEY.md section 6)."""
    if wl["model"] == "burgers":
        return TRUTH - PRIOR_MEAN
    return None


def run_reference(args, wl, name, out_fd):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # bounded sample per bench step, shrunk for long runs so that the whole arm stays within a few minutes
    n = max(1, min(cpu_steps_for(wl), cpu_steps_for(wl) * 7 // max(args.steps, 1)))      # <= ~90 s of chains in total
    u_start = posterior_start(wl)
    for _ in range(args.warmup if args.warmup < 2 else 1):      # process start-up / import warm-up
        cpu_sample(wl, 1, cores, u_start)
    t_busy = 0.0
    steps = accepts = 0
    for _ in range(args.steps):
        v, busy, wall, res = cpu_sample(wl, n, cores, u_start)
        t_busy += busy
        steps += sum(r[1] for r in res)
        accepts += sum(r[2] for r in res)
    value = steps / t_busy
    sample = "%d processes x %d chain-steps per bench step (NumPy restatement, 2 forward solves per step as in the reference)" % (cores, n)
    line = dict(impl="reference", metric="chain_steps_per_sec", value=value, unit="chain-steps/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * t_busy / max(args.steps, 1),
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=workload_config(wl, name, args),
                acceptance_rate=accepts / max(steps, 1),
                cpu_baseline=dict(value=value, unit="chain-steps/s", cores=cores, kind="port", sample=sample,
                                  acceptance=accepts / max(steps, 1)),
                e2e=dict(value=value, unit="chain-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    emit(line, out_fd)


def workload_config(wl, name, args, burn_in=None, start=None):
    cfg = dict(workload=name, chains_per_gpu=wl["chains"], mcmc_steps_per_launch=wl["mcmc_steps"])
    numerics = wl.get("numerics", args.numerics)
    if wl["model"] == "burgers":
        cfg.update(cells=wl["N"], proposer="pCN", beta=wl["beta"], T=1.0, prior="N(u_p, 0.25^2 I_3)",
                   noise_std=0.05, numerics=numerics)
        cfg["untimed_burn_in_steps"] = args.burn_in if burn_in is None else burn_in
        cfg["start"] = start or "u* - prior mean (posterior region), then the untimed burn-in"
    else:
        cfg.update(K=6, J=4, T=wl["T"], proposer="RW", delta=wl["delta"], solves_per_step=2,
                   rtol=1e-3, atol=1e-6, numerics=numerics)
        cfg["untimed_burn_in_steps"] = 0
        cfg["start"] = "the reference's u_0 = (-1.9, 1.9, 0.9) and IC (lorenz_mcmc.py:139), warm-up launches only"
    cfg["l2"] = "flushed between timed launches (256 MiB memset, untimed); working set << L2 anyway"
    cfg["parallelism"] = "chains sharded by global id, dp%d" % args.gpus
    return cfg


# ------------------------------------------------------------------------------------------------
# clocks sampling (NVML) during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index, enabled=True, interval=0.1):
        super().__init__(daemon=True)
        self.interval = interval
        self.samples, self.reasons = [], set()
        self.sm_max = None
        self.stop_flag = False
        self.ok = False
        try:
            if not enabled:
                raise RuntimeError("disabled")
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        while self.ok and not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in {**self.BAD, **self.NOTE}.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.interval)

    def summary(self):
        if not self.samples:
            return None
        return dict(sm_mhz=float(np.median(self.samples)), sm_max_mhz=float(self.sm_max), reasons=sorted(self.reasons),
                    samples=len(self.samples))


# ------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------
def build_problem(M, wl, numerics):
    if wl["model"] == "burgers":
        f = M.BurgersFVM(N=wl["N"], numerics=numerics)
        y = f.at_parameters(TRUTH)           # noise-free synthetic observations G(u*) (burgers_mcmc.py:116)
        prior = M.GaussianDistribution(PRIOR_MEAN, 0.25 ** 2 * np.identity(3))
        pot = M.EvolutionPotential(f, y, M.GaussianDistribution(np.zeros(5), 0.05 ** 2 * np.identity(5)))
        proposer = M.ConstSteppCNProposer(wl["beta"], prior)
        accepter = M.CountedAccepter(M.pCNAccepter(pot))
        u0 = np.zeros(3)
        return pot, proposer, accepter, u0
    g = np.load(os.path.join(ROOT, "tests", "golden", "lorenz_problem_K6_J4.npz"))
    f = M.Lorenz96Moments(6, 4, wl["T"], 1.0, g["prior_means"], g["IC"], numerics=numerics)
    prior = M.GaussianDistribution(np.zeros(3), np.diag([10., 1, 10]))
    pot = M.EvolutionPotential(f, g["y"], M.GaussianDistribution(np.zeros(30), 0.25 * np.diag(g["var"])))
    proposer = M.ConstStepStandardRWProposer(wl["delta"], prior)
    accepter = M.CountedAccepter(M.StandardRWAccepter(pot, prior))
    return pot, proposer, accepter, g["u0"]


def algorithmic_flops(wl, work_a, work_b):
    """SURVEY.md section 8(d): Burgers 29 FLOP per cell per SSPRK2 time step; Lorenz 3444 FLOP per
    Dormand-Prince attempt + 48 per accepted step (K=6, J=4)."""
    if wl["model"] == "burgers":
        return 29.0 * wl["N"] * work_a
    return 3444.0 * (work_a + work_b) + 48.0 * work_a


def last_step_outputs(chains, trace, pooled):
    """Host copies of what the last launch returned (see --dump-outputs).  When the per-chain arrays do not fit
    in DUMP_LIMIT_BYTES, a subset of the chains drawn with a fixed seed is kept."""
    import torch
    per_chain = dict(samples=trace, u=chains.u, phi=chains.phi)
    if chains.model_state is not None:
        per_chain["model_state"] = chains.model_state
    out = {}
    chain_bytes = sum(t[0].numel() * t.element_size() for t in per_chain.values())
    room = DUMP_LIMIT_BYTES - pooled.numel() * pooled.element_size() - 4096     # 4096: the .npy headers
    if chains.n * chain_bytes > room:
        idx = np.sort(np.random.default_rng(0).choice(chains.n, room // (chain_bytes + 8), replace=False))
        sel = torch.as_tensor(idx, device=trace.device)
        per_chain = {k: t.index_select(0, sel) for k, t in per_chain.items()}
        out["chain_index"] = (idx + chains.chain_offset).astype(np.float64)
    out.update({k: t.cpu().numpy() for k, t in per_chain.items()})
    out["pooled"] = pooled.cpu().numpy()
    return out


def write_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype == np.float64, (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def emit(line, out_fd):
    os.write(out_fd, (json.dumps(line) + "\n").encode())


def main():
    # Libraries (NCCL banner, torchrun notes) may write to stdout; the contract is ONE JSON line
    # there.  Keep the real stdout for that line and point fd 1 at stderr for everything else.
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="burgers_pcn_256", choices=sorted(WORKLOADS))
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (default: the workload's)")
    ap.add_argument("--mcmc-steps", type=int, default=0, help="Metropolis steps per launch")
    ap.add_argument("--numerics", default="fused", choices=["exact", "fused"])
    ap.add_argument("--burn-in", type=int, default=1500, help="untimed Metropolis steps before warm-up (Burgers)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workload lines")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the arrays the last timed launch returned to DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    wl = dict(WORKLOADS[args.workload])
    if args.chains:
        wl["chains"] = args.chains
    if args.mcmc_steps:
        wl["mcmc_steps"] = args.mcmc_steps
    if args.impl == "reference":
        return run_reference(args, wl, args.workload, out_fd)

    import torch
    import torch.distributed as dist
    import ip_mcmc_b200 as M
    from ip_mcmc_b200 import parallel
    from ip_mcmc_b200.engine import ChainBatch, F64

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    sm_ghz = torch.cuda.get_device_properties(dev).clock_rate / 1e6 if hasattr(torch.cuda.get_device_properties(dev), "clock_rate") else 1.965
    nominal_fp64 = n_sm * 64 * 2 * 1.965e9 / 1e12      # 64 DFMA lanes per SM per clock at clocks.max.sm

    def measure(wl, K, W, with_e2e=True, trace_chains=64, burn_in=0, start=None, dump=False):
        B, S = wl["chains"], wl["mcmc_steps"]
        pot, proposer, accepter, u0 = build_problem(M, wl, wl.get("numerics", args.numerics))
        sampler = M.MCMCSampler(proposer, accepter, np.random.default_rng(2))
        spec, pot, a = sampler._compile(10 ** 9, 0, 1, None)
        problem = pot.problem()
        if start is not None:
            u0 = start
        chains = ChainBatch(problem, u0, n_chains=B, chain_offset=rank * B)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        trace = torch.empty((B, S, 3), dtype=F64, device=dev)
        kept = []
        if burn_in:                                         # untimed burn-in: leave the prior-mean start
            chains.run(spec, burn_in)
        for _ in range(W):
            chains.run(spec, S, trace=trace)
        torch.cuda.synchronize()
        c0 = chains.counters.sum(0).cpu().numpy()
        # NVML init happens here, before the barrier.  Every rank samples its own GPU (rank 0 at 10 Hz for
        # the contract's `clocks` key, the others at 4 Hz: enough to tell a slow GPU from a slow host)
        sampler_clk = ClockSampler(local, interval=0.02 if rank == 0 else 0.25)
        if world > 1:
            parallel.allreduce_pooled(chains.pooled(), 3)   # warm NCCL with the message of the final reduce
            dist.barrier()
        else:
            chains.pooled()
        torch.cuda.synchronize()
        sampler_clk.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K + 1)]
        launches0 = chains.launches
        if world > 1:
            # align the ranks ON THE DEVICE: the streams wait in a one-element all-reduce until every rank has reached
            # this point, so the host-side skew of eight Python processes (tens of milliseconds: thread start, NVML)
            # does not show up as waiting time in the final collective of the ranks that started early
            dist.all_reduce(torch.zeros(1, dtype=F64, device=dev))
        t_wall0 = time.perf_counter()
        for k in range(K):
            flush.zero_()                                   # evict L2 between timed launches (untimed)
            ev[k][0].record()
            chains.run(spec, S, trace=trace)
            ev[k][1].record()
            kept.append(trace[:trace_chains].clone())
        ev[K][0].record()
        pooled_local = chains.pooled()
        ev_mid = torch.cuda.Event(enable_timing=True)
        ev_mid.record()
        pooled = parallel.allreduce_pooled(pooled_local, 3)  # the only collective of the job (one all-gather)
        ev[K][1].record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
        sampler_clk.stop_flag = True
        sampler_clk.join()
        outputs = last_step_outputs(chains, trace, pooled) if dump else None
        kern_ms = [a.elapsed_time(b) for a, b in ev[:K]]
        red_ms = ev[K][0].elapsed_time(ev[K][1])
        pool_ms = ev[K][0].elapsed_time(ev_mid)
        total_ms = parallel.max_over_ranks(sum(kern_ms) + red_ms, dev)
        clk = sampler_clk.summary() or dict(sm_mhz=float("nan"), reasons=[])
        per_rank = torch.tensor([sum(kern_ms), red_ms, t_wall * 1e3, clk["sm_mhz"], float(len(clk["reasons"])),
                                 max(kern_ms), min(kern_ms)], dtype=F64, device=dev)
        if world > 1:
            gathered = [torch.zeros_like(per_rank) for _ in range(world)]
            dist.all_gather(gathered, per_rank)
            per_rank = torch.stack(gathered)
        per_rank = per_rank.reshape(-1, 7).cpu().numpy().round(3).tolist()
        c1 = chains.counters.sum(0).cpu().numpy()
        dc = (c1 - c0).astype(np.float64)
        cnt = torch.tensor(dc, dtype=F64, device=dev)
        if world > 1:
            dist.all_reduce(cnt)
        dc_all = cnt.cpu().numpy()
        steps_all = B * S * K * world
        value = steps_all / (total_ms * 1e-3)
        # roofline of the dominant (only) kernel, this rank
        flops = algorithmic_flops(wl, dc[2], dc[3])
        achieved = flops / (sum(kern_ms) * 1e-3) / 1e12
        hbm_bytes = B * (2 * 8 * 4 + 8 * 3 * S) * K        # u, Phi in/out + the recorded trace
        tr = torch.stack(kept, dim=1).reshape(min(trace_chains, B), K * S, 3).cpu().numpy()
        ess_tot, ess_per = M.stats.ess_multichain(tr)
        ess_per_chain = ess_tot / tr.shape[0]
        out = dict(value=value, total_ms=total_ms, kern_ms=kern_ms, red_ms=red_ms, pool_ms=pool_ms, per_rank=per_rank, achieved=achieved,
                   hbm_gbs=hbm_bytes / (sum(kern_ms) * 1e-3) / 1e9, counters=dc_all, steps_all=steps_all,
                   acceptance=dc_all[1] / max(dc_all[0], 1), ess_per_sec=ess_per_chain * B * world / (total_ms * 1e-3),
                   ess_per_chain=ess_per_chain, clocks=sampler_clk.summary(), launches=chains.launches - launches0,
                   pooled=pooled.cpu().numpy(), wall_s=t_wall, nonfinite=int(dc_all[4]),
                   mean_work_per_solve=dc_all[2] / max(dc_all[3], 1)
                   if wl["model"] == "burgers" else (dc_all[2] + dc_all[3]) / max(2 * dc_all[0], 1),
                   outputs=outputs)
        if with_e2e:
            # end to end through the public API with HOST buffers: numpy u_0 (and Phi(u_0), known from the run that
            # produced it) in, numpy samples out.  (1) MCMCSampler.run: torch-managed pinned staging;
            # (2) MCMCSampler.run_host = the C entry point ipmcmc_sample_host alone (pageable NumPy buffers).
            u_host = chains.u.cpu().numpy()
            phi_host = None if pot.G.stateful else chains.phi.cpu().numpy()
            ms_host = chains.model_state.cpu().numpy() if chains.model_state is not None else None
            if ms_host is not None:
                pot.G.IC = ms_host[0]
            out_host = torch.empty((B, S, 3), dtype=F64).pin_memory()        # pinned result buffer, reused
            out_np = np.empty((B, S, 3))

            Ke = max(K, 5)      # calls per e2e leg (the 3-step extra workloads: 3 calls were too few for a stable wall clock)

            def timed(fn):
                fn()                                         # warm: allocator, pinned staging, clocks after the host-side ESS
                fn()
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                t0 = time.perf_counter()
                for _ in range(Ke):
                    fn()
                torch.cuda.synchronize()
                return parallel.max_over_ranks((time.perf_counter() - t0) * 1e3, dev)

            dt = timed(lambda: sampler.run(u_host, S, 0, 1, n_chains=B, chain_offset=rank * B, out=out_host, phi_0=phi_host))
            out["e2e"] = dict(value=B * S * Ke * world / (dt * 1e-3), unit="chain-steps/s",
                              h2d_bytes_per_step=int(sampler.last_run["h2d_bytes"]),
                              d2h_bytes_per_step=int(sampler.last_run["d2h_bytes"]),
                              path="MCMCSampler.run(host u_0, Phi(u_0)) -> pinned host samples")
            dt = timed(lambda: sampler.run_host(u_host, S, 0, 1, n_chains=B, chain_offset=rank * B, out=out_np, phi_0=phi_host))
            out["e2e_c_abi"] = dict(value=B * S * Ke * world / (dt * 1e-3), unit="chain-steps/s",
                                    h2d_bytes_per_step=int(sampler.last_run["h2d_bytes"]),
                                    d2h_bytes_per_step=int(sampler.last_run["d2h_bytes"]),
                                    path="ipmcmc_sample_host (ctypes, pageable NumPy buffers, arena + copies inside the C call)")
        return out

    def cold_start(wl, total_steps, reps):
        """The run a user following INTEGRATION.md gets: MCMCSampler.run(u_0 = 0, total_steps, 0, 1) -- ONE
        launch of `total_steps` Metropolis steps per chain from the reference's start (burgers_mcmc.py:129-134),
        no burn-in, all states recorded on the device.  `reps` timed repetitions with different seeds."""
        B = wl["chains"]
        pot, proposer, accepter, u0 = build_problem(M, wl, args.numerics)
        ms, fl, nonfinite, steps_fv, solves = [], [], 0, 0.0, 0.0
        trace = torch.empty((B, total_steps, 3), dtype=F64, device=dev)
        for r in range(reps + 1):                           # first repetition = warm-up (short)
            sampler = M.MCMCSampler(proposer, accepter, np.random.default_rng(100 + r))
            spec, pot, a = sampler._compile(10 ** 9, 0, 1, None)
            chains = ChainBatch(pot.problem(), np.zeros(3), n_chains=B, chain_offset=rank * B)
            n = total_steps if r else min(200, total_steps)
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            chains.run(spec, n, trace=trace[:, :n])
            e1.record()
            torch.cuda.synchronize()
            if r == 0:
                continue
            c = chains.counters.sum(0).double().cpu().numpy()
            ms.append(parallel.max_over_ranks(e0.elapsed_time(e1), dev))
            fl.append(algorithmic_flops(wl, c[2], c[3]) / (e0.elapsed_time(e1) * 1e-3) / 1e12)
            nonfinite += int(c[4])
            steps_fv += c[2]
            solves += c[3]
        tf = float(np.mean(fl))
        return dict(chain_steps_per_sec=B * total_steps * reps * world / (sum(ms) * 1e-3), roofline_tflops=tf,
                    roofline_frac=tf / peak, roofline_frac_nominal=tf / nominal_fp64,
                    ms_per_run=[round(x, 2) for x in ms], slowest_over_fastest=max(ms) / min(ms),
                    nonfinite_phi_per_rank=nonfinite, capped_solves_per_rank=nonfinite,
                    capped_solve_share_of_fv_steps=nonfinite * float(pot.G.effective_max_fv_steps) / max(steps_fv, 1),
                    max_fv_steps=int(pot.G.effective_max_fv_steps),
                    mean_fv_steps_per_solve=steps_fv / max(solves, 1),
                    config=workload_config(wl, args.workload, args, burn_in=0,
                                           start="u_0 = 0 (the reference's start, burgers_mcmc.py:129-134), %d steps "
                                                 "in ONE launch, no burn-in, %d repetitions" % (total_steps, reps)))

    peak = M.fp64_peak_tflops(5)
    # Burgers: every leg (GPU, CPU baseline, --impl reference) measures the STATIONARY phase: chains start
    # in the posterior region (u* - prior mean) and burn in untimed.  The `cold_start` leg measures the run from
    # the reference's u_0 = 0 without any burn-in.
    burn_in, start = (args.burn_in if wl['model'] == 'burgers' else 0), None
    if wl['model'] == 'burgers':
        start = TRUTH - PRIOR_MEAN
        if wl['N'] >= 1024:
            burn_in = min(burn_in, 200)        # a solve costs ~30 MFLOP here: keep the untimed part short
    args.burn_in = burn_in
    res = measure(wl, args.steps, max(args.warmup, 3), burn_in=burn_in, start=start,
                  dump=bool(args.dump_outputs) and rank == 0)
    if res["outputs"] is not None:
        write_outputs(args.dump_outputs, res["outputs"])
    extra = {}
    cold = None
    if not args.no_extra and args.workload == "burgers_pcn_256":
        # the other BASELINE.json configs, at EVERY N (weak scaling: the same per-GPU batch on every rank)
        plan = [("lorenz_rw", dict(WORKLOADS["lorenz_rw"]), 0, True),
                ("burgers_pcn_1024", dict(WORKLOADS["burgers_pcn_1024"]), 100, False),
                ("burgers_pcn_256_exact", dict(WORKLOADS["burgers_pcn_256"], numerics="exact", mcmc_steps=200), 400, False)]
        for name, w, b_in, e2e in plan:
            r = measure(w, 3, 3, with_e2e=e2e, trace_chains=8, burn_in=b_in,
                        start=(TRUTH - PRIOR_MEAN) if w["model"] == "burgers" else None)
            extra[name] = dict(chain_steps_per_sec=r["value"], acceptance=r["acceptance"],
                               roofline_tflops=r["achieved"], roofline_frac=r["achieved"] / peak,
                               roofline_frac_nominal=r["achieved"] / nominal_fp64, ms_per_step=r["total_ms"] / 3,
                               allreduce_ms=r["red_ms"], pool_moments_ms=r["pool_ms"], nonfinite_phi=r["nonfinite"],
                               per_rank_ms=dict(columns=["sum_kernel", "final_reduce", "wall_timed_region", "sm_mhz",
                                                         "n_throttle_reasons", "slowest_launch", "fastest_launch"],
                                                rows=r["per_rank"]),
                               config=workload_config(w, name, args, burn_in=b_in))
            for k in ("e2e", "e2e_c_abi"):
                if k in r:
                    extra[name][k] = r[k]
        cold = cold_start(dict(wl), 5000, 3)
    short = None
    if not args.no_extra and args.workload == "burgers_pcn_256" and wl["mcmc_steps"] > SHORT_LAUNCH_STEPS:
        # the same workload in 200-step launches (what rounds 1 and 2a timed): the launch tail is paid 5x as often
        r = measure(dict(wl, mcmc_steps=SHORT_LAUNCH_STEPS), 5, 3, with_e2e=False, trace_chains=8, burn_in=burn_in, start=start)
        short = dict(chain_steps_per_sec=r["value"], roofline_tflops=r["achieved"], roofline_frac=r["achieved"] / peak,
                     roofline_frac_nominal=r["achieved"] / nominal_fp64, ms_per_step=r["total_ms"] / 5,
                     mcmc_steps_per_launch=SHORT_LAUNCH_STEPS)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[args.workload]["traffic"]
    except Exception:
        pass
    roofline = dict(bound="fp64", achieved=res["achieved"], peak=peak, unit="TFLOP/s", frac=res["achieved"] / peak,
                    traffic=traffic, peak_nominal=nominal_fp64, frac_of_nominal=res["achieved"] / nominal_fp64,
                    peak_source="DFMA micro-benchmark (ipmcmc_fp64_peak) measured in this run; MEASURED_PEAKS.json has "
                                "no fp64 entry; peak_nominal = %d SM x 64 FMA/clk x 2 x 1.965 GHz" % n_sm,
                    flops_model="29 FLOP per cell per SSPRK2 step x device-counted FV steps" if wl["model"] == "burgers"
                    else "3444 FLOP per RK45 attempt x device-counted attempts",
                    hbm=dict(achieved=res["hbm_gbs"], peak=hbm_peak, unit="GB/s", frac=res["hbm_gbs"] / hbm_peak,
                             peak_source="MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"))
    line = dict(metric="chain_steps_per_sec", value=res["value"], unit="chain-steps/s", n_gpus=world, steps=args.steps,
                warmup=max(args.warmup, 3), ms_per_step=res["total_ms"] / args.steps, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=workload_config(wl, args.workload, args), roofline=roofline, e2e=res.get("e2e"),
                e2e_c_abi=res.get("e2e_c_abi"),
                gpu_launches=int(res["launches"]), clocks=res["clocks"], ess_per_sec=res["ess_per_sec"],
                ess_per_chain_in_timed_window=res["ess_per_chain"], acceptance_rate=res["acceptance"],
                nonfinite_phi=res["nonfinite"],
                mean_work_per_solve=res["mean_work_per_solve"], allreduce_ms=res["red_ms"], pool_moments_ms=res["pool_ms"],
                kernel_ms_per_step=[round(x, 3) for x in res["kern_ms"]],
                per_rank_ms=dict(columns=["sum_kernel", "final_reduce", "wall_timed_region", "sm_mhz", "n_throttle_reasons",
                                          "slowest_launch", "fastest_launch"], rows=res["per_rank"]),
                posterior_mean=[float(x) for x in res["pooled"][1:4]], cold_start=cold, short_launch=short,
                extra_workloads=extra)
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        line.update(cpu_baselines(wl, cores))
        if not args.no_extra:
            for name in ("lorenz_rw", "burgers_pcn_1024"):
                if name in extra:
                    extra[name].update(cpu_baselines(dict(WORKLOADS[name]), cores))
    emit(line, out_fd)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
