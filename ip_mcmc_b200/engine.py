"""Thin object layer over the C ABI: problem handles and batched chain state in torch buffers.

PyTorch is used only for device memory and streams; all arithmetic happens in libipmcmc.so.
There is no CPU path: constructing a Problem without a CUDA device or without the built library
raises.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check

F64 = torch.float64


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.EngineError("no CUDA device: ip_mcmc_b200 runs on sm_100a only (no CPU fallback)")


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def potential_tables(data, noise_distribution):
    """Constant tables of Phi(u) = -noise.logpdf(data - G(u)) (potential.py:53-54)."""
    y = np.ascontiguousarray(np.asarray(data, dtype=np.float64).reshape(-1))
    q = y.shape[0]
    if noise_distribution is None:
        return dict(q=q, y=y, dense=False, perm=np.arange(q, dtype=np.int32), scale=np.ones(q), LP=None,
                    log_const=0.0)
    if noise_distribution.k != q:
        raise ValueError("noise dimension %d != data dimension %d" % (noise_distribution.k, q))
    if np.any(noise_distribution.mean != 0):
        # logpdf(y - G) with mean m equals the zero-mean logpdf of (y - m) - G
        y = y - noise_distribution.mean
    LP, log_pdet, rank = noise_distribution.whitener()
    log_const = rank * np.log(2 * np.pi) + log_pdet
    nz = LP != 0
    if np.all(nz.sum(axis=0) == 1):
        # one non-zero per column: diagonal covariance, columns possibly permuted by eigh
        perm = np.argmax(nz, axis=0).astype(np.int32)
        scale = LP[perm, np.arange(q)].copy()
        return dict(q=q, y=y, dense=False, perm=perm, scale=scale, LP=None, log_const=float(log_const))
    return dict(q=q, y=y, dense=True, perm=None, scale=None, LP=np.ascontiguousarray(LP), log_const=float(log_const))


def _fill_potential(desc, tab, keep):
    desc.n_obs = tab["q"]
    desc.whiten_dense = 1 if tab["dense"] else 0
    desc.y = _lib.as_double_p(tab["y"])
    keep.append(tab["y"])
    if tab["dense"]:
        desc.LP = _lib.as_double_p(tab["LP"])
        keep.append(tab["LP"])
    else:
        perm = np.ascontiguousarray(tab["perm"], dtype=np.int32)
        scale = np.ascontiguousarray(tab["scale"], dtype=np.float64)
        desc.perm = _lib.as_int32_p(perm)
        desc.scale = _lib.as_double_p(scale)
        keep += [perm, scale]
    desc.log_const = tab["log_const"]


class Problem:
    """A forward model + Gaussian-misfit potential resident on the current CUDA device."""

    def __init__(self, model, data=None, noise_distribution=None):
        _require_cuda()
        self.lib = _lib.load()
        self.model = model
        self.kind = model.kind
        self.d = model.n_params
        self.q = model.n_obs
        if data is None:
            data = np.zeros(self.q)
        tab = potential_tables(data, noise_distribution)
        if tab["q"] != self.q:
            raise ValueError("data has %d entries, the observation operator returns %d" % (tab["q"], self.q))
        keep = []
        handle = C.c_void_p()
        if self.kind == _lib.MODEL_BURGERS:
            desc = model._c_desc(keep)
            _fill_potential(desc.potential, tab, keep)
            check(self.lib.ipmcmc_burgers_create(C.byref(desc), C.byref(handle)))
            self.state_size = model.N
        else:
            desc = model._c_desc(keep)
            _fill_potential(desc.potential, tab, keep)
            check(self.lib.ipmcmc_lorenz_create(C.byref(desc), C.byref(handle)))
            self.state_size = model.n_var
        self.handle = handle
        self.device = torch.device("cuda", torch.cuda.current_device())

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self.lib.ipmcmc_destroy(h)
            self.handle = None

    # ---- batched forward evaluation (ipmcmc_forward) -------------------------------------------
    def forward(self, u, state=None, want_state=False):
        """u: [n, d] (numpy or cuda tensor).  Returns dict(G [n,q], phi [n], work [n,2], state).
        Lorenz: `state` [n, n_var] is the initial condition (required) and is returned advanced."""
        u_t = torch.as_tensor(np.asarray(u, dtype=np.float64) if not torch.is_tensor(u) else u,
                              dtype=F64, device=self.device).reshape(-1, self.d).contiguous()
        n = u_t.shape[0]
        G = torch.empty((n, self.q), dtype=F64, device=self.device)
        phi = torch.empty((n,), dtype=F64, device=self.device)
        work = torch.zeros((n, 2), dtype=torch.int64, device=self.device)
        st = None
        if self.kind == _lib.MODEL_LORENZ:
            if state is None:
                raise ValueError("Lorenz forward needs the initial condition `state` [n, n_var]")
            st = torch.as_tensor(np.asarray(state, dtype=np.float64) if not torch.is_tensor(state) else state,
                                 dtype=F64, device=self.device).reshape(n, self.state_size).clone()
        elif want_state:
            st = torch.empty((n, self.state_size), dtype=F64, device=self.device)
        check(self.lib.ipmcmc_forward(self.handle, n, _ptr(u_t), _ptr(G), _ptr(phi), _ptr(st), _ptr(work), _stream()))
        return dict(G=G, phi=phi, work=work, state=st)


class ChainBatch:
    """State of `n_chains` independent chains on the device (u, Phi(u), carried model state,
    Welford moments, counters)."""

    COUNTER_NAMES = ("calls", "accepts", "work_a", "work_b", "nonfinite", "constraint_rejects")

    def __init__(self, problem, u0, n_chains=None, model_state=None, chain_offset=0, phi0=None):
        self.problem = problem
        dev = problem.device
        d = problem.d
        u0 = np.asarray(u0, dtype=np.float64) if not torch.is_tensor(u0) else u0
        u0_t = torch.as_tensor(u0, dtype=F64)
        if u0_t.ndim == 1:
            if n_chains is None:
                n_chains = 1
            u0_t = u0_t.reshape(1, d).expand(n_chains, d)
        elif n_chains is None:
            n_chains = u0_t.shape[0]
        if tuple(u0_t.shape) != (n_chains, d):
            raise ValueError("u_0 has shape %s, expected (%d,) or (%d, %d)" % (tuple(u0_t.shape), d, n_chains, d))
        self.n = int(n_chains)
        self.d = d
        self.chain_offset = int(chain_offset)
        if u0_t.device.type != "cuda":
            u0_t = u0_t.contiguous().pin_memory()
        self.u = u0_t.to(dev, non_blocking=True).contiguous().clone()
        self.h2d_bytes = self.u.numel() * 8
        if phi0 is None:
            # NaN = not evaluated yet: the first launch solves for Phi(u_0)
            self.phi = torch.full((self.n,), float("nan"), dtype=F64, device=dev)
        else:
            # Phi(u_0) known (e.g. `last_run["phi"]` of the run that produced u_0): no extra solve
            ph = torch.as_tensor(np.asarray(phi0, dtype=np.float64) if not torch.is_tensor(phi0) else phi0, dtype=F64)
            if ph.numel() != self.n:
                raise ValueError("phi0 has %d entries, expected %d" % (ph.numel(), self.n))
            if ph.device.type != "cuda":
                ph = ph.contiguous().pin_memory()
            self.phi = ph.reshape(self.n).to(dev, non_blocking=True).contiguous().clone()
            self.h2d_bytes += self.n * 8
        self.model_state = None
        if problem.kind == _lib.MODEL_LORENZ:
            ms = problem.model.IC if model_state is None else model_state
            ms_t = torch.as_tensor(np.asarray(ms, dtype=np.float64) if not torch.is_tensor(ms) else ms, dtype=F64)
            if ms_t.ndim == 1:
                ms_t = ms_t.reshape(1, -1).expand(self.n, -1)
            if tuple(ms_t.shape) != (self.n, problem.state_size):
                raise ValueError("model state has shape %s" % (tuple(ms_t.shape),))
            if ms_t.device.type != "cuda":
                ms_t = ms_t.contiguous().pin_memory()
            self.model_state = ms_t.to(dev, non_blocking=True).contiguous().clone()
            self.h2d_bytes += self.model_state.numel() * 8
        self.mom_count = torch.zeros((self.n,), dtype=F64, device=dev)
        self.mom_mean = torch.zeros((self.n, d), dtype=F64, device=dev)
        self.mom_m2 = torch.zeros((self.n, d), dtype=F64, device=dev)
        self.counters = torch.zeros((self.n, _lib.N_COUNTERS), dtype=torch.int64, device=dev)
        self.step = 0
        self._keep = []
        self._pool_scratch = None
        self.launches = 0
        # optional [n_chains] float64 cuda tensor: inverse temperature of each chain's likelihood (replica
        # exchange, tempering.py); None runs the untempered kernel path (ipmcmc_run)
        self.inv_temp = None
        self.sched = None          # scratch of the dynamic step scheduler (Burgers N <= 1024 and d <= 32, Lorenz)
        self.sched_chunk = 0       # Metropolis steps per work item; 0 = automatic (Burgers: min(4, max(1, n_steps // 64)); Lorenz: 1)
        if problem.kind == _lib.MODEL_LORENZ or (problem.model.N <= 1024 and d <= _lib.MAX_DIM):
            self.sched = torch.empty((3 * self.n + 2,), dtype=torch.int64, device=dev)

    def run(self, spec, n_steps, trace=None, steplog=None, vlog=None, inject_w=None, inject_u=None):
        """Advance all chains by n_steps in ONE launch of the fused kernel (ipmcmc_run).
        spec: SamplerSpec.  trace: optional cuda tensor [n, n_record, d] for recorded samples."""
        lib = self.problem.lib
        s = spec.c_desc(self, n_steps)
        b = _lib.ChainBuffers()
        b.u_dev = _ptr(self.u)
        b.phi_dev = _ptr(self.phi)
        b.model_state_dev = _ptr(self.model_state)
        b.mom_count_dev = _ptr(self.mom_count)
        b.mom_mean_dev = _ptr(self.mom_mean)
        b.mom_m2_dev = _ptr(self.mom_m2)
        b.counters_dev = _ptr(self.counters)
        b.trace_dev = _ptr(trace)
        b.n_record = 0 if trace is None else trace.shape[1]
        b.steplog_dev = _ptr(steplog)
        b.vlog_dev = _ptr(vlog)
        b.inject_w_dev = _ptr(inject_w)
        b.inject_u_dev = _ptr(inject_u)
        if self.sched is not None:
            b.sched_dev = _ptr(self.sched)
            b.sched_len = self.sched.numel()
        b.sched_chunk = self.sched_chunk
        if self.inv_temp is None:
            check(lib.ipmcmc_run(self.problem.handle, C.byref(s), C.byref(b), self.n, int(n_steps), _stream()))
        else:
            check(lib.ipmcmc_run_tempered(self.problem.handle, C.byref(s), C.byref(b), _ptr(self._inv_temp_checked()),
                                          self.n, int(n_steps), _stream()))
        self.step += int(n_steps)
        self.launches += 1

    def _inv_temp_checked(self):
        t = self.inv_temp
        if not (torch.is_tensor(t) and t.dtype == F64 and t.device == self.u.device and t.is_contiguous()
                and t.numel() == self.n):
            raise ValueError("inv_temp must be a contiguous float64 tensor of %d entries on %s" % (self.n, self.u.device))
        return t

    def swap(self, ladder_size, seed, round, replica, swap_counts, round_trips, inject_u=None):
        """One replica-exchange round between adjacent rungs of the batch's ladders (ipmcmc_swap_replicas): the
        batch is n / ladder_size ladders, ladder-major, tempered by `inv_temp`.  replica [n, 2] int32, swap_counts
        [n_ladders, ladder_size - 1, 2] int64 and round_trips [n_ladders] int64 are updated in place; inject_u
        [n_ladders, ladder_size - 1] replaces the Philox swap uniforms."""
        K = int(ladder_size)
        if K < 2 or self.n % K:
            raise ValueError("%d chains do not form ladders of %d rungs" % (self.n, K))
        L = self.n // K
        for name, x, shape, dt in (("replica", replica, (self.n, 2), torch.int32),
                                   ("swap_counts", swap_counts, (L, K - 1, 2), torch.int64),
                                   ("round_trips", round_trips, (L,), torch.int64),
                                   ("inject_u", inject_u, (L, K - 1), F64)):
            if x is not None and (tuple(x.shape) != shape or x.dtype != dt or not x.is_contiguous()
                                  or x.device != self.u.device):
                raise ValueError("%s must be a contiguous %s tensor of shape %s on %s" % (name, dt, shape, self.u.device))
        check(self.problem.lib.ipmcmc_swap_replicas(L, K, self.d, _ptr(self.u), _ptr(self.phi),
                                                    _ptr(self._inv_temp_checked()), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                    self.chain_offset, int(round), _ptr(inject_u), _ptr(replica),
                                                    _ptr(swap_counts), _ptr(round_trips), _stream()))
        self.launches += 1

    def pooled(self):
        """Chan-merged moments + counters over this batch: cuda tensor [2d + 7]
        (n, mean[d], M2[d], calls, accepts, work_a, work_b, nonfinite, constraint_rejects)."""
        lib = self.problem.lib
        out = torch.empty((2 * self.d + 1 + _lib.N_COUNTERS,), dtype=F64, device=self.problem.device)
        if self._pool_scratch is None:
            nbytes = int(lib.ipmcmc_pool_scratch_bytes(self.n, self.d))
            self._pool_scratch = torch.empty((max(nbytes, 8),), dtype=torch.uint8, device=self.problem.device)
        check(lib.ipmcmc_pool_moments(self.n, self.d, _ptr(self.mom_count), _ptr(self.mom_mean), _ptr(self.mom_m2),
                                      _ptr(self.counters), _ptr(out), _ptr(self._pool_scratch),
                                      self._pool_scratch.numel(), _stream()))
        self.launches += 2
        return out


class SamplerSpec:
    """Host description of proposer + accepter, compiled from the reference-style objects."""

    def __init__(self, dim, proposer_kind, accepter_kind, coef_u=1.0, coef_w=0.0, schedule=None, factor=None,
                 prior_chol=None, constraint=None, recompute_phi_u=False, seed=0, record_start=0,
                 record_interval=1):
        self.dim = int(dim)
        self.proposer_kind = int(proposer_kind)
        self.accepter_kind = int(accepter_kind)
        self.coef_u, self.coef_w = float(coef_u), float(coef_w)
        self.schedule = None if schedule is None else np.ascontiguousarray(schedule, dtype=np.float64)
        self.schedule_dev = None
        self.schedule_origin = 0       # global step index of schedule row 0
        self.factor = None
        self.factor_kind = 0
        if factor is not None:
            f = np.asarray(factor, dtype=np.float64)
            if f.ndim == 2 and np.all((f != 0).sum(axis=1) == 1) and np.all((f != 0).sum(axis=0) == 1):
                # diagonal covariance: numpy's SVD factor is a scaled signed permutation of z.  The z_i
                # are iid Philox normals, so w_i = f_i * z_i has the same law without the permutation.
                f = f[np.arange(f.shape[0]), np.argmax(f != 0, axis=1)].copy()
            if f.ndim == 1 and np.all(f == 1.0):
                self.factor_kind = 0
            else:
                self.factor_kind = 1 if f.ndim == 1 else 2
                self.factor = np.ascontiguousarray(f)
        self.prior_chol = None if prior_chol is None else np.ascontiguousarray(prior_chol, dtype=np.float64)
        self.constraint = constraint
        self.recompute_phi_u = bool(recompute_phi_u)
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.record_start = int(record_start)
        self.record_interval = int(record_interval)

    def c_desc(self, chains, n_steps):
        s = _lib.SamplerDesc()
        keep = chains._keep
        del keep[:]
        s.dim = self.dim
        s.proposer = self.proposer_kind
        s.accepter = self.accepter_kind
        s.factor_kind = self.factor_kind
        s.recompute_phi_u = 1 if self.recompute_phi_u else 0
        s.coef_u, s.coef_w = self.coef_u, self.coef_w
        if self.schedule is not None:
            if self.schedule_dev is None:
                self.schedule_dev = torch.as_tensor(self.schedule, dtype=F64).to(chains.problem.device)
            # rows are indexed by the GLOBAL step number: shift the base pointer by the origin
            s.coef_sched_dev = self.schedule_dev.data_ptr() - 16 * self.schedule_origin
            s.n_sched = self.schedule.shape[0] + self.schedule_origin
        if self.factor is not None:
            s.factor = _lib.as_double_p(self.factor)
        if self.prior_chol is not None:
            s.prior_chol = _lib.as_double_p(self.prior_chol)
        if self.constraint is not None:
            c = self.constraint
            lo = np.ascontiguousarray(np.broadcast_to(c.lo, (self.dim,)), dtype=np.float64)
            hi = np.ascontiguousarray(np.broadcast_to(c.hi, (self.dim,)), dtype=np.float64)
            sh = np.ascontiguousarray(np.broadcast_to(c.shift, (self.dim,)), dtype=np.float64)
            keep += [lo, hi, sh]
            s.has_constraint = 1
            s.box_lo, s.box_hi, s.box_shift = _lib.as_double_p(lo), _lib.as_double_p(hi), _lib.as_double_p(sh)
        s.seed = self.seed
        s.chain_offset = chains.chain_offset
        s.first_step = chains.step
        s.record_start = self.record_start
        s.record_interval = self.record_interval
        return s


def fp64_peak_tflops(iters=5):
    """Measured dependent-free DFMA throughput of the current device (roofline denominator)."""
    _require_cuda()
    out = C.c_double()
    check(_lib.load().ipmcmc_fp64_peak(iters, C.byref(out)))
    return out.value
