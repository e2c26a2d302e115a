// Lorenz kernels: batched forward evaluation, the fused Metropolis kernel, and the RHS / single
// RK-attempt probes used by the parity tests.  floor(32/K) chains per warp.
#pragma once
#include "lorenz.cuh"
#include "sampler.cuh"
#include "sched.cuh"

namespace ipmcmc {

// smem per CTA: (groups + 1 dummy) x (G[MAX_OBS] | r2[MAX_OBS])
__host__ __device__ inline int lorenz_groups(int K) { return 32 / K; }
__host__ __device__ inline size_t lorenz_smem_bytes(int K) {
    return (size_t)(lorenz_groups(K) + 1) * 2 * IPMCMC_MAX_OBS * sizeof(double);
}
// warps per CTA whose shared memory fits the default dynamic shared-memory limit of 48 KB
inline int lorenz_warps_fit(int K) { return (int)((48 * 1024) / lorenz_smem_bytes(K)); }

template <int J, int KT, int NUM>
__device__ __forceinline__ void lorenz_load_state(const LorenzLanes<J, KT, NUM> &L, const double *s, double (&y)[J + 1]) {
    y[0] = s[L.k];
#pragma unroll
    for (int j = 0; j < J; ++j) y[1 + j] = s[L.K + L.k * J + j];
}
template <int J, int KT, int NUM>
__device__ __forceinline__ void lorenz_store_state(const LorenzLanes<J, KT, NUM> &L, double *s, const double (&y)[J + 1]) {
    s[L.k] = y[0];
#pragma unroll
    for (int j = 0; j < J; ++j) s[L.K + L.k * J + j] = y[1 + j];
}

// LorenzObservationOperator.__call__ (lorenz_mcmc.py:55-68) + EvolutionPotential (potential.py:53-54)
// for every chain of the warp at once.  `ui`: component i of the chain's u on group lane i.
// S.y carries the initial condition in and the end state out (lorenz_mcmc.py:66).
template <int J, int KT, int NUM>
__device__ __forceinline__ double lorenz_phi(const LorenzLanes<J, KT, NUM> &L, const LorenzDev &P, double ui,
                                          LorenzSolve<J, KT, NUM> &S,
                                          bool active, double *Gs, double *r2) {
    // F, h, b = prior_means + u   (lorenz_mcmc.py:64)
    const double pi = (L.k < 3) ? P.param_mean[L.k] + ui : 0.0;
    LorenzTheta th;
    th.F = __shfl_sync(FULL, pi, L.base + 0);
    th.h = __shfl_sync(FULL, pi, L.base + 1);
    th.b = __shfl_sync(FULL, pi, L.base + 2);
    th.c = P.c;
    th.finish(J);
    double ykeep[J + 1];
#pragma unroll
    for (int i = 0; i < J + 1; ++i) ykeep[i] = S.y[i];
    S.solve(L, P, th, active);
    if (!active) {  // an inactive chain keeps its state
#pragma unroll
        for (int i = 0; i < J + 1; ++i) S.y[i] = ykeep[i];
    }
    // np.mean(moment_function(y), axis=1)   (lorenz_mcmc.py:68)
    const double nt = (double)S.n_t;
#pragma unroll
    for (int m = 0; m < 5; ++m) Gs[m * L.K + L.k] = S.msum[m] / nt;
    __syncwarp();
    return potential_from_G(P.pot, Gs, r2, L.k, L.K, FULL);
}

template <int J, int KT, int NUM>
__global__ void __launch_bounds__(256, 1) lorenz_forward_kernel(const __grid_constant__ LorenzDev P, long long n,
                                                            const double *__restrict__ u, double *__restrict__ G,
                                                            double *__restrict__ phi, double *__restrict__ state,
                                                            long long *__restrict__ work) {
    extern __shared__ double smem_all[];
    const int lane = lane_id();
    const int groups = lorenz_groups(P.K);
    // W warps per CTA (warp w sits on SM sub-partition w % 4); warps never synchronise with each other
    const int warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    double *smem = smem_all + (size_t)warp * (lorenz_smem_bytes(P.K) / sizeof(double));
    LorenzLanes<J, KT, NUM> L;
    L.init(lane, P.K, groups);
    const int slot = L.valid ? lane / P.K : groups;
    double *Gs = smem + (size_t)slot * 2 * IPMCMC_MAX_OBS, *r2 = Gs + IPMCMC_MAX_OBS;
    for (long long c0 = ((long long)blockIdx.x * wpc + warp) * groups; c0 < n; c0 += (long long)gridDim.x * wpc * groups) {
        const long long c = c0 + slot;
        const bool active = L.valid && c < n;
        LorenzSolve<J, KT, NUM> S;
#pragma unroll
        for (int i = 0; i < J + 1; ++i) S.y[i] = 0.0;
        if (active) lorenz_load_state<J, KT, NUM>(L, state + c * P.nvar, S.y);
        const double ui = (active && L.k < 3) ? u[c * 3 + L.k] : 0.0;
        const double ph = lorenz_phi<J, KT, NUM>(L, P, ui, S, active, Gs, r2);
        if (active) {
            lorenz_store_state<J, KT, NUM>(L, state + c * P.nvar, S.y);
            if (G)
                for (int i = L.k; i < P.pot.q; i += P.K) G[c * P.pot.q + i] = Gs[i];
            if (L.k == 0) {
                if (phi) phi[c] = ph;
                if (work) {
                    work[2 * c] = S.n_acc;
                    work[2 * c + 1] = S.n_rej;
                }
            }
        }
        __syncwarp();
    }
}

// Metropolis steps [s0, s1) of the launch for the warp's group of chains c0 .. c0 + groups - 1
// (chain c0 + slot on this lane group): load the chain state, step, store it back.  Another SM may have
// written the state earlier in the launch (sched.cuh): it is read and written through L2.
template <int J, int KT, int NUM>
__device__ __forceinline__ void lorenz_advance_group(const LorenzDev &P, const SamplerDev &Sd, const ChainBufDev &C,
                                                     const LorenzLanes<J, KT, NUM> &L, const Group &Gp, int slot,
                                                     double *Gs, double *r2, long long n_chains, long long n_steps,
                                                     long long c0, long long s0, long long s1) {
    const int d = Sd.d;  // 3
    const long long c = c0 + slot;
    const bool active = L.valid && c < n_chains;
    const long long cs = active ? c : 0;  // safe index for predicated-off lanes
    const long long cg = Sd.chain_offset + cs;
    const bool own = active && L.k < d;
    LorenzSolve<J, KT, NUM> S;
#pragma unroll
    for (int i = 0; i < J + 1; ++i) S.y[i] = 0.0;
    if (active) {
        const double *ms = C.model_state + c * P.nvar;
        S.y[0] = __ldcg(ms + L.k);
#pragma unroll
        for (int j = 0; j < J; ++j) S.y[1 + j] = __ldcg(ms + L.K + L.k * J + j);
    }
    double ui = own ? __ldcg(C.u + c * d + L.k) : 0.0;
    double phi_u = active ? __ldcg(C.phi + c) : 0.0;
    long long cnt[CNT_N];
#pragma unroll
    for (int k = 0; k < CNT_N; ++k) cnt[k] = 0;
    double reg_u = (Sd.accepter == IPMCMC_ACCEPT_RW) ? prior_regulariser(Sd, Gp, ui) : 0.0;
    Welford mom{active ? __ldcg(C.mom_count + c) : 0.0, own ? __ldcg(C.mom_mean + c * d + L.k) : 0.0,
                own ? __ldcg(C.mom_m2 + c * d + L.k) : 0.0};
    long long n_rec = recorded_before(Sd, Sd.first_step + s0) - recorded_before(Sd, Sd.first_step);

    for (long long s = s0; s < s1; ++s) {
        const long long gstep = Sd.first_step + s;
        double ca, cb;
        step_coefs(Sd, gstep, ca, cb);
        const double w = proposal_noise(Sd, C, Gp, cs, cg, s, n_steps, gstep);
        const double vi = ca * ui + cb * w;
        if (C.vlog && own) C.vlog[(c * n_steps + s) * d + L.k] = vi;
        // the box test ballots over the FULL warp: every lane evaluates it, `active` is applied afterwards
        const bool cok = !Sd.has_constraint || constraint_ok(Sd, Gp, vi);
        const bool ok = active && cok;
        // The reference evaluates Phi(u) and then Phi(v) every step, each solve starting where
        // the previous one ended (accepter.py:121-122 + lorenz_mcmc.py:66).  One inlined call
        // site serves both passes so the integrator state stays in registers.
        const bool need_u = ok && (Sd.recompute_phi_u || isnan(phi_u));
        double ph_v = 0.0;
        for (int pass = __any_sync(FULL, need_u) ? 0 : 1; pass < 2; ++pass) {
            const bool act = pass ? ok : need_u;
            const double ph = lorenz_phi<J, KT, NUM>(L, P, pass ? vi : ui, S, act, Gs, r2);
            if (act) {
                if (pass) ph_v = ph; else phi_u = ph;
                if (!pass) {
                    cnt[CNT_WORK_A] += S.n_acc;
                    cnt[CNT_WORK_B] += S.n_rej;
                }
            }
        }
        bool accepted = false;
        double phi_v = nan(""), a = nan("");
        int work = 0;
        if (ok) {
            phi_v = ph_v;
            work = S.n_acc + S.n_rej;
            cnt[CNT_WORK_A] += S.n_acc;
            cnt[CNT_WORK_B] += S.n_rej;
        }
        double reg_v = 0.0;
        if (Sd.accepter == IPMCMC_ACCEPT_RW) reg_v = prior_regulariser(Sd, Gp, vi);
        if (ok) {
            a = exp((phi_u + reg_u) - (phi_v + reg_v));
            const double U = C.inject_u ? C.inject_u[c * n_steps + s]
                                        : draw_uniform(Sd.seed, (uint64_t)cg, (uint64_t)gstep);
            accepted = a > U;
            if (!isfinite(phi_v)) cnt[CNT_NONFINITE] += 1;
            if (accepted) {
                ui = vi;
                phi_u = phi_v;
                reg_u = reg_v;
            }
        } else if (active) {
            cnt[CNT_CONSTRAINT] += 1;
        }
        cnt[CNT_CALLS] += 1;
        cnt[CNT_ACCEPTS] += accepted ? 1 : 0;
        if (C.steplog && active && L.k == 0) {
            double *Lg = C.steplog + (c * n_steps + s) * 4;
            Lg[0] = phi_v;
            Lg[1] = a;
            Lg[2] = accepted ? 1.0 : 0.0;
            Lg[3] = (double)work;
        }
        if (records_step(Sd, gstep)) {
            mom.add(ui);
            if (C.trace && n_rec < C.n_record && own) C.trace[(c * C.n_record + n_rec) * d + L.k] = ui;
            ++n_rec;
        }
    }
    if (active) {
        double *ms = C.model_state + c * P.nvar;
        __stcg(ms + L.k, S.y[0]);
#pragma unroll
        for (int j = 0; j < J; ++j) __stcg(ms + L.K + L.k * J + j, S.y[1 + j]);
        if (own) {
            __stcg(C.u + c * d + L.k, ui);
            __stcg(C.mom_mean + c * d + L.k, mom.mean);
            __stcg(C.mom_m2 + c * d + L.k, mom.m2);
        }
        if (L.k == 0) {
            __stcg(C.phi + c, phi_u);
            __stcg(C.mom_count + c, mom.count);
            // a chain belongs to one warp at a time: read-modify-write through L2 needs no atomic
#pragma unroll
            for (int k = 0; k < CNT_N; ++k)
                __stcg(C.counters + c * CNT_N + k, __ldcg(C.counters + c * CNT_N + k) + cnt[k]);
        }
    }
    __syncwarp();
}

// Dynamic step scheduler (sched.cuh): the work unit is a warp's group of floor(32/K) chains, an item is
// `chunk` Metropolis steps of it.  With 820 warps on 592 sub-partitions (4096 chains, K = 6) a static map
// leaves the sub-partitions that hold one warp idle for ~45 % of the launch; rotating the groups over the
// warps lets every group advance at the average pace.
template <int J, int KT, int NUM>
__global__ void __launch_bounds__(256, 1) lorenz_chain_queue_kernel(const __grid_constant__ LorenzDev P,
                                                                const __grid_constant__ SamplerDev Sd,
                                                                const __grid_constant__ ChainBufDev C,
                                                                long long n_chains, long long n_steps, int chunk) {
    extern __shared__ double smem_all[];
    const int lane = lane_id();
    const int groups = lorenz_groups(P.K);
    const int warp = threadIdx.x >> 5;
    double *smem = smem_all + (size_t)warp * (lorenz_smem_bytes(P.K) / sizeof(double));
    LorenzLanes<J, KT, NUM> L;
    L.init(lane, P.K, groups);
    const int slot = L.valid ? lane / P.K : groups;
    double *Gs = smem + (size_t)slot * 2 * IPMCMC_MAX_OBS, *r2 = Gs + IPMCMC_MAX_OBS;
    const Group Gp{L.base, P.K, L.k, FULL};
    const long long n_units = (n_chains + groups - 1) / groups;
    // the launch spreads ceil(n_units / n_CTA) warps per CTA over ALL SMs (engine.cu); the surplus warps of
    // the last rows leave at once instead of spinning on an empty queue beside a working warp
    if ((long long)warp * gridDim.x + blockIdx.x >= n_units) return;
    sched_serve(C.sched, n_units, n_steps, chunk, lane, [&](long long g, long long s0, long long s1) {
        lorenz_advance_group<J, KT, NUM>(P, Sd, C, L, Gp, slot, Gs, r2, n_chains, n_steps, g * groups, s0, s1);
    });
}

// ---- probes -------------------------------------------------------------------------------
template <int J, int KT, int NUM>
__global__ void __launch_bounds__(32) lorenz_rhs_kernel(int K, long long n, const double *__restrict__ theta,
                                                        const double *__restrict__ state, double *__restrict__ out) {
    const int lane = lane_id();
    const int groups = lorenz_groups(K);
    const int nvar = K * (J + 1);
    LorenzLanes<J, KT, NUM> L;
    L.init(lane, K, groups);
    const int slot = L.valid ? lane / K : groups;
    for (long long c0 = (long long)blockIdx.x * groups; c0 < n; c0 += (long long)gridDim.x * groups) {
        const long long c = c0 + slot;
        const bool active = L.valid && c < n;
        double y[J + 1], dy[J + 1];
#pragma unroll
        for (int i = 0; i < J + 1; ++i) y[i] = 0.0;
        LorenzTheta th{0, 0, 0, 0, 0, 0};
        if (active) {
            lorenz_load_state<J, KT, NUM>(L, state + c * nvar, y);
            th = LorenzTheta{theta[4 * c], theta[4 * c + 1], theta[4 * c + 2], theta[4 * c + 3], 0, 0};
        }
        th.finish(J);
        L.to_scaled(th, y);      // FUSED numerics: the right-hand side of the scaled fast variables (lorenz.cuh)
        L.rhs(th, y, dy);
        L.from_scaled(th, dy);
        if (active) lorenz_store_state<J, KT, NUM>(L, out + c * nvar, dy);
    }
}

template <int J, int KT, int NUM>
__global__ void __launch_bounds__(32) lorenz_attempt_kernel(int K, long long n, const double *__restrict__ theta,
                                                            const double *__restrict__ state,
                                                            const double *__restrict__ hstep, double rtol, double atol,
                                                            double *__restrict__ out) {
    const int lane = lane_id();
    const int groups = lorenz_groups(K);
    const int nvar = K * (J + 1);
    LorenzLanes<J, KT, NUM> L;
    L.init(lane, K, groups);
    const int slot = L.valid ? lane / K : groups;
    const double inv_sqrt_n = 1.0 / sqrt((double)nvar);
    for (long long c0 = (long long)blockIdx.x * groups; c0 < n; c0 += (long long)gridDim.x * groups) {
        const long long c = c0 + slot;
        const bool active = L.valid && c < n;
        double y[J + 1], f[J + 1], yn[J + 1], fn[J + 1];
#pragma unroll
        for (int i = 0; i < J + 1; ++i) y[i] = 0.0;
        LorenzTheta th{0, 0, 0, 0, 0, 0};
        double h = 0.0;
        if (active) {
            lorenz_load_state<J, KT, NUM>(L, state + c * nvar, y);
            th = LorenzTheta{theta[4 * c], theta[4 * c + 1], theta[4 * c + 2], theta[4 * c + 3], 0, 0};
            h = hstep[c];
        }
        th.finish(J);
        L.to_scaled(th, y);
        L.rhs(th, y, f);
        double ss;
        if (NUM == LNUM_FUSED) {
            double ys2[J + 1];
            L.stage2(y, f, h, ys2);
            ss = L.attempt_fused(th, y, f, ys2, h, rtol, atol, atol * fabs(th.s), yn, fn);
        } else {
            ss = L.attempt(th, y, f, h, rtol, atol, yn, fn);
        }
        L.from_scaled(th, yn);
        L.from_scaled(th, fn);
        const double err = sqrt(ss) * inv_sqrt_n;
        if (active) {
            double *o = out + c * (2 * nvar + 1);
            lorenz_store_state<J, KT, NUM>(L, o, yn);
            lorenz_store_state<J, KT, NUM>(L, o + nvar, fn);
            if (L.k == 0) o[2 * nvar] = err;
        }
    }
}

}  // namespace ipmcmc
