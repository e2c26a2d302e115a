// Burgers kernels: batched forward evaluation and the fused Metropolis kernel.
// One chain per warp, one warp per CTA (the hardware block scheduler then balances the
// data-dependent solve lengths across the 148 SMs); the FV state never leaves registers, the end
// state is staged once per solve in shared memory for the windowed trapezoid measurement.
#pragma once
#include "burgers.cuh"
#include "burgers_team.cuh"
#include "sampler.cuh"
#include "sched.cuh"

// Register budget of the static chain kernel: 128 registers (2 CTAs of 256 threads per SM) up to 8 cells
// per lane, 255 from 16 cells per lane on, where 128 spill the state (measured: burgers_launch_impl.cuh,
// burgers_launch_chain_queue).
#ifndef IPMCMC_CHAIN_MINB
#define IPMCMC_CHAIN_MINB(CPL) ((CPL) >= 16 ? 1 : 2)
#endif

namespace ipmcmc {

// shared memory layout per warp: state[N] | G[MAX_OBS] | r2[MAX_OBS]
__host__ __device__ inline size_t burgers_smem_bytes(int N, int warps = 1) {
    return (size_t)warps * (N + 2 * IPMCMC_MAX_OBS) * sizeof(double);
}

// Measurer.__call__ (utilities.py:100-109): m_i = 10 * trapz(values[l:r], dx) with numpy's
// evaluation (dx*(y[1:]+y[:-1])/2.0).sum() in pairwise order; lane i handles window i.
__device__ __forceinline__ void burgers_measure(const BurgersDev &B, const double *state, double *Gs, int lane) {
    for (int i = lane; i < B.pot.q; i += 32) {
        const int l = B.win_left[i], r = B.win_right[i];
        const int nterm = r - l - 1;
        double sum = 0.0;
        if (nterm >= 1) {
            const double dxm = B.dx_meas;
            sum = np_pairwise_sum([&](int j) { return dxm * (state[j + 1] + state[j]) / 2.0; }, l, nterm);
        }
        Gs[i] = 10.0 * sum;
    }
    __syncwarp();
}

// G and Phi of the absolute parameters `param`, given as BurgersWarp::integrate takes them: parameter i on
// lane i (d <= 32) or a ParamAt functor (d > 32).  Leaves the end state in smem `state` and G in `Gs`.
// Returns Phi; n_fv by reference.
template <int CPL, int NUMERICS, bool PADDED, class Param>
__device__ __forceinline__ double burgers_solve_phi(const BurgersDev &B, const Param &param, double *state, double *Gs,
                                                   double *r2, int lane, int &n_fv) {
    BurgersWarp<CPL, NUMERICS, PADDED> W;
    PROF_T(p0);
    n_fv = W.integrate(B, param, lane);
    PROF_T(p1);
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
        const int c = lane * CPL + k;
        if (c < B.N) state[c] = W.u[k];
    }
    __syncwarp();
    burgers_measure(B, state, Gs, lane);
    const double phi = potential_from_G(B.pot, Gs, r2, lane, 32, FULL);
    PROF_T(p2);
    PROF_ADD(3, p0, p1);   // -DIPMCMC_PROF builds: every Burgers one-warp solve, the wide path's included
    PROF_ADD(4, p1, p2);
    // a solve stopped by the safety cap has not reached T: report it as non-finite (-> rejected)
    return W.capped ? nan("") : phi;
}

// G(u) and Phi(u) for the parameter vector whose component i sits on lane i (value `ui`).
// Inlined at its call sites on purpose: with the solve as an out-of-line subroutine ptxas allocates the
// time-step loop's registers around the call convention and schedules it measurably worse (B200,
// 1024 x 256 cells: 60 % of the fp64 peak out of line, 66 % inlined; 8192 x 1024: 78 % / 83 %).
#ifndef IPMCMC_PHI_INLINE
#define IPMCMC_PHI_INLINE __forceinline__
#endif
template <int CPL, int NUMERICS, bool PADDED>
__device__ IPMCMC_PHI_INLINE double burgers_phi(const BurgersDev &B, double ui, double *state, double *Gs, double *r2,
                                              int lane, int &n_fv) {
    // FVMObservationOperator.__call__ (utilities.py:40-41): IC(u_0 + u)
    const double pi = (lane < B.d) ? B.param_mean[lane] + ui : 0.0;
    return burgers_solve_phi<CPL, NUMERICS, PADDED>(B, pi, state, Gs, r2, lane, n_fv);
}

// Outputs of forward evaluation c (null pointers are skipped): G and the end state from shared memory,
// Phi and the work.  Thread t of the nt threads that evaluated it (a warp or a team) writes every nt-th value.
__device__ __forceinline__ void burgers_store_forward(const BurgersDev &B, long long c, const double *Gs,
                                                      const double *state, double ph, int n_fv, double *G, double *phi,
                                                      double *state_out, long long *work, int t, int nt) {
    if (G)
        for (int i = t; i < B.pot.q; i += nt) G[c * B.pot.q + i] = Gs[i];
    if (state_out)
        for (int i = t; i < B.N; i += nt) state_out[c * B.N + i] = state[i];
    if (t == 0) {
        if (phi) phi[c] = ph;
        if (work) {
            work[2 * c] = n_fv;
            work[2 * c + 1] = 0;
        }
    }
}

template <int CPL, int NUMERICS, bool PADDED>
__global__ void __launch_bounds__(256) burgers_forward_kernel(const __grid_constant__ BurgersDev B, long long n,
                                                              const double *__restrict__ u, double *__restrict__ G,
                                                              double *__restrict__ phi, double *__restrict__ state_out,
                                                              long long *__restrict__ work) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    double *smem = smem_all + (size_t)warp * (B.N + 2 * IPMCMC_MAX_OBS);
    double *state = smem, *Gs = smem + B.N, *r2 = Gs + IPMCMC_MAX_OBS;
    const int lane = lane_id();
    for (long long c = (long long)blockIdx.x * wpc + warp; c < n; c += (long long)gridDim.x * wpc) {
        const double ui = (lane < B.d) ? u[c * B.d + lane] : 0.0;
        int n_fv;
        const double ph = burgers_phi<CPL, NUMERICS, PADDED>(B, ui, state, Gs, r2, lane, n_fv);
        burgers_store_forward(B, c, Gs, state, ph, n_fv, G, phi, state_out, work, lane, 32);
        __syncwarp();
    }
}

// The chain's parameter vector u and its proposal v, component i on lane i (d <= 32): u and its Welford moments
// in registers, v a register value; the free functions of sampler.cuh (shared with the Lorenz kernels) do the work.
struct LaneVec {
    double u;
    Welford mom;

    // v = ca*u + cb*w (proposer.py:29-30, 81-82), logged to vlog
    __device__ __forceinline__ double propose(const SamplerDev &S, const ChainBufDev &C, const Group &Gp, long long c,
                                              long long cg, long long s, long long n_steps, long long gstep, double ca,
                                              double cb, bool writer) const {
        const double w = proposal_noise(S, C, Gp, c, cg, s, n_steps, gstep);
        const double v = ca * u + cb * w;
        if (writer && C.vlog && Gp.lane < S.d) C.vlog[(c * n_steps + s) * S.d + Gp.lane] = v;
        return v;
    }
    __device__ __forceinline__ bool inside(const SamplerDev &S, const Group &Gp, double x) const {
        return constraint_ok(S, Gp, x);
    }
    __device__ __forceinline__ double regulariser(const SamplerDev &S, const Group &Gp, double x) const {
        return prior_regulariser(S, Gp, x);
    }
    __device__ __forceinline__ void accept(const SamplerDev &, const Group &, double v) { u = v; }
    // recorded sample n_rec of the launch: moments, trace
    __device__ __forceinline__ void record(const SamplerDev &S, const ChainBufDev &C, const Group &Gp, long long c,
                                           long long n_rec, bool writer) {
        mom.add(u);
        if (writer && C.trace && n_rec < C.n_record && Gp.lane < S.d) C.trace[(c * C.n_record + n_rec) * S.d + Gp.lane] = u;
    }
    template <bool QUEUE>
    __device__ __forceinline__ void load_u(const SamplerDev &S, const ChainBufDev &C, int lane, long long c) {
        u = (lane < S.d) ? ld_state<QUEUE>(C.u + c * S.d + lane) : 0.0;
    }
    template <bool QUEUE>
    __device__ __forceinline__ void load_moments(const SamplerDev &S, const ChainBufDev &C, int lane, long long c) {
        const int d = S.d;
        mom = Welford{ld_state<QUEUE>(C.mom_count + c), (lane < d) ? ld_state<QUEUE>(C.mom_mean + c * d + lane) : 0.0,
                      (lane < d) ? ld_state<QUEUE>(C.mom_m2 + c * d + lane) : 0.0};
    }
    // u and the per-component moments; the count is stored by lane 0 (count())
    template <bool QUEUE>
    __device__ __forceinline__ void store(const SamplerDev &S, const ChainBufDev &C, int lane, long long c) const {
        const int d = S.d;
        if (lane < d) {
            st_state<QUEUE>(C.u + c * d + lane, u);
            st_state<QUEUE>(C.mom_mean + c * d + lane, mom.mean);
            st_state<QUEUE>(C.mom_m2 + c * d + lane, mom.m2);
        }
    }
    __device__ __forceinline__ double count() const { return mom.count; }
};

// Registers of one chain between Metropolis steps.  `Vec`: where its parameter vector lives, LaneVec or
// SmemVec (wide path).
template <class Vec>
struct ChainRegs {
    Vec x;
    double phi_u, reg_u;
    long long cnt[CNT_N];
};

// ONE Metropolis step of chain c (local id; cg global id) at launch-local step s: proposal -> (box
// constraint) -> solve -> Phi(v) -> accept/reject -> counters, logs, moments, trace.
// `phi_of(x, n_fv)` evaluates Phi for a parameter vector of R's kind (R.x.u or the proposal): the one-warp
// solver (burgers_phi), the multi-warp team solver (burgers_team_phi), whose warps all run this same step
// with the same Philox draws, or the one-warp solver over a shared-memory vector (burgers_phi_wide); `writer`
// (warp 0 of a team; always true for one warp per chain) owns the global-memory outputs.
#ifndef IPMCMC_STEP_INLINE
#define IPMCMC_STEP_INLINE __forceinline__
#endif
template <class Vec, class PhiOf>
__device__ IPMCMC_STEP_INLINE void metropolis_step(const SamplerDev &S, const ChainBufDev &C, const Group &Gp, long long c,
                                                   long long cg, long long s, long long n_steps, ChainRegs<Vec> &R,
                                                   const PhiOf &phi_of, bool writer) {
    const int lane = Gp.lane;
    const long long gstep = S.first_step + s;
    double ca, cb;
    PROF_T(q0);
    step_coefs(S, gstep, ca, cb);
    const auto v = R.x.propose(S, C, Gp, c, cg, s, n_steps, gstep, ca, cb, writer);
    PROF_T(q1);
    PROF_ADD(2, q0, q1);
    bool accepted = false;
    double phi_v = nan(""), a = nan("");
    int n_fv = 0;
    const bool ok = !S.has_constraint || R.x.inside(S, Gp, v);
    if (ok) {
        if (S.recompute_phi_u) {  // the reference's 2 solves per step (accepter.py:121-122)
            int nf0;
            R.phi_u = phi_of(R.x.u, nf0);
            R.cnt[CNT_WORK_A] += nf0;
            R.cnt[CNT_WORK_B] += 1;
        }
        phi_v = phi_of(v, n_fv);
        PROF_T(q2);
        R.cnt[CNT_WORK_A] += n_fv;
        R.cnt[CNT_WORK_B] += 1;
        double reg_v = 0.0;
        if (S.accepter == IPMCMC_ACCEPT_RW) reg_v = R.x.regulariser(S, Gp, v);
        // the chain's inverse temperature t tempers Phi, not the RW regulariser; Phi itself stays untempered.  t = 1
        // (every untempered chain) multiplies exactly: the reference's exp((Phi(u)+reg_u) - (Phi(v)+reg_v)).  Read
        // here, after the solve, rather than carried in ChainRegs: a register live across the solve moves its allocation.
        const double t = C.inv_temp ? C.inv_temp[c] : 1.0;
        a = exp((t * R.phi_u + R.reg_u) - (t * phi_v + reg_v));
        const double U = C.inject_u ? C.inject_u[c * n_steps + s] : draw_uniform(S.seed, (uint64_t)cg, (uint64_t)gstep);
        accepted = a > U;  // strict, un-clipped; NaN compares false (accepter.py:61-62)
        if (!isfinite(phi_v)) R.cnt[CNT_NONFINITE] += 1;
        if (accepted) {
            R.x.accept(S, Gp, v);
            R.phi_u = phi_v;
            R.reg_u = reg_v;
        }
        PROF_T(q3);
        PROF_ADD(5, q2, q3);
    } else {
        R.cnt[CNT_CONSTRAINT] += 1;
    }
    R.cnt[CNT_CALLS] += 1;
    R.cnt[CNT_ACCEPTS] += accepted ? 1 : 0;
    if (writer && C.steplog && lane == 0) {
        double *L = C.steplog + (c * n_steps + s) * 4;
        L[0] = phi_v;
        L[1] = a;
        L[2] = accepted ? 1.0 : 0.0;
        L[3] = (double)n_fv;
    }
    // recording (sampler.py:23-28)
    if (records_step(S, gstep)) R.x.record(S, C, Gp, c, recorded_before(S, gstep) - recorded_before(S, S.first_step), writer);
}

// Chain c's registers from global memory (ld_state<QUEUE>); `x` says where the parameter vector goes.  On the
// chain's first launch Phi(u_0) is not known yet (NaN) and is solved for with `phi_of`.  `team`: every warp of
// the CTA runs this for the same chain, and all must have read the state before warp 0 may overwrite it
// (burgers_store_chain).
template <bool QUEUE, class Vec, class PhiOf>
__device__ __forceinline__ ChainRegs<Vec> burgers_load_chain(const SamplerDev &S, const ChainBufDev &C, const Group &Gp,
                                                             long long c, const Vec &x, const PhiOf &phi_of, bool team) {
    ChainRegs<Vec> R{x};
    R.x.template load_u<QUEUE>(S, C, Gp.lane, c);
    R.phi_u = ld_state<QUEUE>(C.phi + c);
#pragma unroll
    for (int k = 0; k < CNT_N; ++k) R.cnt[k] = 0;
    if (team) __syncthreads();
    if (isnan(R.phi_u)) {
        int n_fv;
        R.phi_u = phi_of(R.x.u, n_fv);
        R.cnt[CNT_WORK_A] += n_fv;
        R.cnt[CNT_WORK_B] += 1;
    }
    R.reg_u = (S.accepter == IPMCMC_ACCEPT_RW) ? R.x.regulariser(S, Gp, R.x.u) : 0.0;
    R.x.template load_moments<QUEUE>(S, C, Gp.lane, c);
    return R;
}

// Chain c's registers back to global memory; the counters accumulate over launches.  A chain belongs to
// one warp (or team) at a time, so their read-modify-write needs no atomic, under the queue too (sched.cuh).
template <bool QUEUE, class Vec>
__device__ __forceinline__ void burgers_store_chain(const SamplerDev &S, const ChainBufDev &C, int lane, long long c,
                                                    const ChainRegs<Vec> &R) {
    R.x.template store<QUEUE>(S, C, lane, c);
    if (lane == 0) {
        st_state<QUEUE>(C.phi + c, R.phi_u);
        st_state<QUEUE>(C.mom_count + c, R.x.count());
#pragma unroll
        for (int k = 0; k < CNT_N; ++k)
            st_state<QUEUE>(C.counters + c * CNT_N + k, ld_state<QUEUE>(C.counters + c * CNT_N + k) + R.cnt[k]);
    }
}

// `phi_of` of the one-warp solver.  A functor and not a lambda: with three call sites (first launch, Phi(u),
// Phi(v)) NVVM outlined a lambda's call operator, and with it the whole solve (see burgers_phi).
template <int CPL, int NUMERICS, bool PADDED>
struct BurgersPhiOf {
    const BurgersDev &B;
    double *state, *Gs, *r2;
    int lane;
    __device__ __forceinline__ double operator()(double ui, int &n_fv) const {
        return burgers_phi<CPL, NUMERICS, PADDED>(B, ui, state, Gs, r2, lane, n_fv);
    }
};

// Metropolis steps [s0, s1) of the launch for chain c on one warp: load the chain state into `x`, step, store it back.
template <bool QUEUE, class Vec, class PhiOf>
__device__ __forceinline__ void burgers_advance_chain(const SamplerDev &S, const ChainBufDev &C, const Group &Gp,
                                                      long long c, long long s0, long long s1, long long n_steps,
                                                      const Vec &x, const PhiOf &phi_of) {
    const long long cg = S.chain_offset + c;
    ChainRegs<Vec> R = burgers_load_chain<QUEUE>(S, C, Gp, c, x, phi_of, false);
    for (long long s = s0; s < s1; ++s) metropolis_step(S, C, Gp, c, cg, s, n_steps, R, phi_of, true);
    burgers_store_chain<QUEUE>(S, C, Gp.lane, c, R);
    __syncwarp();
}

// W warps per CTA, one chain per warp.  Warps never synchronise with each other; the CTA shape
// only pins which chains share an SM sub-partition (warp w -> SMSP w % 4).
template <int CPL, int NUMERICS, bool PADDED>
__global__ void __launch_bounds__(256, IPMCMC_CHAIN_MINB(CPL)) burgers_chain_kernel(const __grid_constant__ BurgersDev B,
                                                            const __grid_constant__ SamplerDev S,
                                                            const __grid_constant__ ChainBufDev C, long long n_chains,
                                                            long long n_steps) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    double *smem = smem_all + (size_t)warp * (B.N + 2 * IPMCMC_MAX_OBS);
    double *state = smem, *Gs = smem + B.N, *r2 = Gs + IPMCMC_MAX_OBS;
    const Group Gp{0, 32, lane_id(), FULL};
    const long long n_slots = C.slot_chain ? (long long)C.n_slots : n_chains;
    for (long long slot = (long long)blockIdx.x * wpc + warp; slot < n_slots; slot += (long long)gridDim.x * wpc) {
        const long long c = C.slot_chain ? (long long)C.slot_chain[slot] : slot;
        if (c < 0 || c >= n_chains) continue;
        burgers_advance_chain<false>(S, C, Gp, c, 0, n_steps, n_steps, LaneVec{},
                                     BurgersPhiOf<CPL, NUMERICS, PADDED>{B, state, Gs, r2, Gp.lane});
    }
}

// Dynamic step scheduler (sched.cuh): the work unit is a chain, an item is `chunk` Metropolis steps of it.
// MINB: register budget, 2 = 128 registers (16 warps per SM), 1 = 255 registers; chosen by the number of
// cells per lane in burgers_launch_chain_queue (burgers_launch_impl.cuh), where the measurements are quoted.
template <int CPL, int NUMERICS, bool PADDED, int MINB>
__global__ void __launch_bounds__(256, MINB) burgers_chain_queue_kernel(
    const __grid_constant__ BurgersDev B, const __grid_constant__ SamplerDev S, const __grid_constant__ ChainBufDev C,
    long long n_chains, long long n_steps, int chunk) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5;
    double *smem = smem_all + (size_t)warp * (B.N + 2 * IPMCMC_MAX_OBS);
    double *state = smem, *Gs = smem + B.N, *r2 = Gs + IPMCMC_MAX_OBS;
    const int lane = lane_id();
    const Group Gp{0, 32, lane, FULL};
    sched_serve(C.sched, n_chains, n_steps, chunk, lane, [&](long long c, long long s0, long long s1) {
        burgers_advance_chain<true>(S, C, Gp, c, s0, s1, n_steps, LaneVec{},
                                    BurgersPhiOf<CPL, NUMERICS, PADDED>{B, state, Gs, r2, lane});
    });
}

// ------------------------------------------------------------------------------------------------
// wide parameter vectors (IPMCMC_MAX_DIM < d <= IPMCMC_MAX_DIM_WIDE): the truncated KL / spectral prior
// with up to 253 modes.  One chain per warp as before, but the parameter vector no longer fits the lanes
// of the warp: u, the proposal v and the absolute parameters live in shared memory (component i is served
// by lane i % 32), the solver reads its parameters from there (BurgersWarp::integrate over a ParamAt
// functor).  The chain runs the same metropolis_step, burgers_load_chain and burgers_store_chain as the
// one-warp kernels, over SmemVec instead of LaneVec: same Philox draws (slot = component), same accept rule;
// diagonal sampling factor and diagonal prior factor only (what a KL prior is); static chain -> warp map.
// CPU statement: oracle/mcmc_np.run_chain + oracle/burgers_np with kl_basis.
// ------------------------------------------------------------------------------------------------
// shared memory per warp: state[N] | G[MAX_OBS] | r2[MAX_OBS] | par[d] | u[d] | v[d]
__host__ __device__ inline size_t burgers_wide_smem_bytes(int N, int d, int warps = 1) {
    return (size_t)warps * (N + 2 * IPMCMC_MAX_OBS + 3 * d) * sizeof(double);
}

// Phi for the parameter perturbation x[0..d) (shared memory); par[] is scratch for mean + x
template <int CPL, int NUMERICS, bool PADDED>
__device__ __forceinline__ double burgers_phi_wide(const BurgersDev &B, const double *x, double *par, double *state,
                                                   double *Gs, double *r2, int lane, int &n_fv) {
    for (int i = lane; i < B.d; i += 32) par[i] = B.param_mean_wide[i] + x[i];   // utilities.py:41
    __syncwarp();
    return burgers_solve_phi<CPL, NUMERICS, PADDED>(B, [par](int i) { return par[i]; }, state, Gs, r2, lane, n_fv);
}

// `phi_of` of the one-warp solver over a shared-memory parameter vector; a functor for the reason given at
// BurgersPhiOf.
template <int CPL, int NUMERICS, bool PADDED>
struct BurgersWidePhiOf {
    const BurgersDev &B;
    double *par, *state, *Gs, *r2;
    int lane;
    __device__ __forceinline__ double operator()(const double *x, int &n_fv) const {
        return burgers_phi_wide<CPL, NUMERICS, PADDED>(B, x, par, state, Gs, r2, lane, n_fv);
    }
};

// The chain's parameter vector u and its proposal v in shared memory, component i on lane i % 32 (d > 32).
// The Welford moments are updated in place in global memory, their count is kept in a register.
struct SmemVec {
    double *u, *v;   // [d] each, in the warp's shared memory
    double n;        // Welford count

    // v = ca*u + cb*w (proposer.py:29-30, 81-82), w_i = factor_i * z_i, z_i = Philox slot i; logged to vlog
    __device__ __forceinline__ const double *propose(const SamplerDev &S, const ChainBufDev &C, const Group &Gp,
                                                     long long c, long long cg, long long s, long long n_steps,
                                                     long long gstep, double ca, double cb, bool writer) const {
        const int d = S.d;
        for (int i = Gp.lane; i < d; i += 32) {
            double w;
            if (C.inject_w) {
                w = C.inject_w[(c * n_steps + s) * d + i];
            } else {
                const double z = draw_normal(S.seed, (uint64_t)cg, (uint64_t)gstep, (uint32_t)i);
                w = S.factor_kind == 1 ? S.factor[i] * z : z;
            }
            const double vi = ca * u[i] + cb * w;
            v[i] = vi;
            if (writer && C.vlog) C.vlog[(c * n_steps + s) * d + i] = vi;
        }
        __syncwarp();
        return v;
    }
    // the box lo | hi | shift from the device table S.box_wide; all lanes agree
    __device__ __forceinline__ bool inside(const SamplerDev &S, const Group &Gp, const double *x) const {
        const int d = S.d;
        bool in = true;
        for (int i = Gp.lane; i < d; i += 32) {
            const double sh = x[i] + S.box_wide[2 * d + i];
            in = in && (sh > S.box_wide[i]) && (sh < S.box_wide[d + i]);
        }
        return __all_sync(FULL, in);
    }
    // 0.5 * ||L x||^2 for a diagonal L (accepter.py:104-106)
    __device__ __forceinline__ double regulariser(const SamplerDev &S, const Group &Gp, const double *x) const {
        const int d = S.d;
        double ss = 0.0;
        for (int i = Gp.lane; i < d; i += 32) {
            const double y = S.prior_chol_diag[i] * x[i];
            ss = ss + y * y;
        }
        const double nrm = sqrt(warp_sum_fixed(ss));
        return 0.5 * (nrm * nrm);
    }
    __device__ __forceinline__ void accept(const SamplerDev &S, const Group &Gp, const double *x) {
        const int d = S.d;
        for (int i = Gp.lane; i < d; i += 32) u[i] = x[i];
        __syncwarp();
    }
    // recorded sample n_rec of the launch: Welford in place, trace
    __device__ __forceinline__ void record(const SamplerDev &S, const ChainBufDev &C, const Group &Gp, long long c,
                                           long long n_rec, bool writer) {
        const int d = S.d;
        n += 1.0;
        for (int i = Gp.lane; i < d; i += 32) {
            const double x = u[i], m0 = C.mom_mean[c * d + i];
            const double delta = x - m0, m1 = m0 + delta / n;
            C.mom_mean[c * d + i] = m1;
            C.mom_m2[c * d + i] += delta * (x - m1);
            if (writer && C.trace && n_rec < C.n_record) C.trace[(c * C.n_record + n_rec) * d + i] = x;
        }
    }
    template <bool QUEUE>
    __device__ __forceinline__ void load_u(const SamplerDev &S, const ChainBufDev &C, int lane, long long c) {
        const int d = S.d;
        // unrolled by 4 as the compiler unrolled these copies when they were written out in the kernel: fewer
        // spills in the wide kernels (ptxas -v)
#pragma unroll 4
        for (int i = lane; i < d; i += 32) u[i] = ld_state<QUEUE>(C.u + c * d + i);
        __syncwarp();
    }
    template <bool QUEUE>
    __device__ __forceinline__ void load_moments(const SamplerDev &, const ChainBufDev &C, int, long long c) {
        n = ld_state<QUEUE>(C.mom_count + c);
    }
    template <bool QUEUE>
    __device__ __forceinline__ void store(const SamplerDev &S, const ChainBufDev &C, int lane, long long c) const {
        const int d = S.d;
#pragma unroll 4
        for (int i = lane; i < d; i += 32) st_state<QUEUE>(C.u + c * d + i, u[i]);
    }
    __device__ __forceinline__ double count() const { return n; }
};

template <int CPL, int NUMERICS, bool PADDED>
__global__ void __launch_bounds__(128) burgers_wide_forward_kernel(const __grid_constant__ BurgersDev B, long long n,
                                                                   const double *__restrict__ u, double *__restrict__ G,
                                                                   double *__restrict__ phi, double *__restrict__ state_out,
                                                                   long long *__restrict__ work) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5, wpc = blockDim.x >> 5, d = B.d;
    double *smem = smem_all + (size_t)warp * (B.N + 2 * IPMCMC_MAX_OBS + 3 * d);
    double *state = smem, *Gs = smem + B.N, *r2 = Gs + IPMCMC_MAX_OBS, *par = r2 + IPMCMC_MAX_OBS, *x = par + d;
    const int lane = lane_id();
    for (long long c = (long long)blockIdx.x * wpc + warp; c < n; c += (long long)gridDim.x * wpc) {
        for (int i = lane; i < d; i += 32) x[i] = u[c * d + i];
        __syncwarp();
        int n_fv;
        const double ph = burgers_phi_wide<CPL, NUMERICS, PADDED>(B, x, par, state, Gs, r2, lane, n_fv);
        burgers_store_forward(B, c, Gs, state, ph, n_fv, G, phi, state_out, work, lane, 32);
        __syncwarp();
    }
}

template <int CPL, int NUMERICS, bool PADDED>
__global__ void __launch_bounds__(128) burgers_wide_chain_kernel(const __grid_constant__ BurgersDev B,
                                                                 const __grid_constant__ SamplerDev S,
                                                                 const __grid_constant__ ChainBufDev C, long long n_chains,
                                                                 long long n_steps) {
    extern __shared__ double smem_all[];
    const int warp = threadIdx.x >> 5, wpc = blockDim.x >> 5, d = S.d;
    double *smem = smem_all + (size_t)warp * (B.N + 2 * IPMCMC_MAX_OBS + 3 * d);
    double *state = smem, *Gs = smem + B.N, *r2 = Gs + IPMCMC_MAX_OBS, *par = r2 + IPMCMC_MAX_OBS, *us = par + d, *vs = us + d;
    const Group Gp{0, 32, lane_id(), FULL};
    const BurgersWidePhiOf<CPL, NUMERICS, PADDED> phi_of{B, par, state, Gs, r2, Gp.lane};
    for (long long c = (long long)blockIdx.x * wpc + warp; c < n_chains; c += (long long)gridDim.x * wpc)
        burgers_advance_chain<false>(S, C, Gp, c, 0, n_steps, n_steps, SmemVec{us, vs}, phi_of);
}

// ------------------------------------------------------------------------------------------------
// team kernels: one CTA of TM warps per chain (N = TM*32*CPL cells > 1024)
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline size_t burgers_team_smem_bytes(int N) {
    return sizeof(TeamXch) + (size_t)(N + 2 * IPMCMC_MAX_OBS) * sizeof(double);
}

// Every warp of the team calls this with the same ui; warp 0 measures and evaluates Phi, the value is
// broadcast through shared memory so that all warps take the same accept decision.
template <int CPL, int NUMERICS, int TM>
__device__ __noinline__ double burgers_team_phi(const BurgersDev &B, TeamXch &X, double ui, double *state, double *Gs,
                                                double *r2, int tw, int lane, int &n_fv) {
    const double pi = (lane < B.d) ? B.param_mean[lane] + ui : 0.0;
    BurgersTeam<CPL, NUMERICS, TM> W;
    n_fv = W.integrate(B, X, pi, tw, lane);
#pragma unroll
    for (int k = 0; k < CPL; ++k) state[(tw * 32 + lane) * CPL + k] = W.u[k];
    __syncthreads();
    if (tw == 0) {
        burgers_measure(B, state, Gs, lane);
        const double phi = potential_from_G(B.pot, Gs, r2, lane, 32, FULL);
        if (lane == 0) X.phi = W.capped ? nan("") : phi;
    }
    __syncthreads();
    return X.phi;
}

template <int CPL, int NUMERICS, int TM>
__global__ void __launch_bounds__(32 * TM) burgers_team_forward_kernel(const __grid_constant__ BurgersDev B, long long n,
                                                                      const double *__restrict__ u,
                                                                      double *__restrict__ G, double *__restrict__ phi,
                                                                      double *__restrict__ state_out,
                                                                      long long *__restrict__ work) {
    extern __shared__ double smem_all[];
    TeamXch &X = *reinterpret_cast<TeamXch *>(smem_all);
    double *state = smem_all + sizeof(TeamXch) / sizeof(double), *Gs = state + B.N, *r2 = Gs + IPMCMC_MAX_OBS;
    const int tw = threadIdx.x >> 5, lane = lane_id();
    for (long long c = blockIdx.x; c < n; c += gridDim.x) {
        const double ui = (lane < B.d) ? u[c * B.d + lane] : 0.0;
        int n_fv;
        const double ph = burgers_team_phi<CPL, NUMERICS, TM>(B, X, ui, state, Gs, r2, tw, lane, n_fv);
        burgers_store_forward(B, c, Gs, state, ph, n_fv, G, phi, state_out, work, threadIdx.x, blockDim.x);
        __syncthreads();
    }
}

template <int CPL, int NUMERICS, int TM>
__global__ void __launch_bounds__(32 * TM) burgers_team_chain_kernel(const __grid_constant__ BurgersDev B,
                                                                    const __grid_constant__ SamplerDev S,
                                                                    const __grid_constant__ ChainBufDev C,
                                                                    long long n_chains, long long n_steps) {
    extern __shared__ double smem_all[];
    TeamXch &X = *reinterpret_cast<TeamXch *>(smem_all);
    double *state = smem_all + sizeof(TeamXch) / sizeof(double), *Gs = state + B.N, *r2 = Gs + IPMCMC_MAX_OBS;
    const int tw = threadIdx.x >> 5, lane = lane_id();
    const bool writer = tw == 0;  // all warps run the same Metropolis logic; warp 0 owns the global writes
    const Group Gp{0, 32, lane, FULL};
    const auto phi_of = [&](double ui, int &n_fv) {
        return burgers_team_phi<CPL, NUMERICS, TM>(B, X, ui, state, Gs, r2, tw, lane, n_fv);
    };
    for (long long c = blockIdx.x; c < n_chains; c += gridDim.x) {
        const long long cg = S.chain_offset + c;
        ChainRegs<LaneVec> R = burgers_load_chain<false>(S, C, Gp, c, LaneVec{}, phi_of, true);
        for (long long s = 0; s < n_steps; ++s) metropolis_step(S, C, Gp, c, cg, s, n_steps, R, phi_of, writer);
        __syncthreads();
        if (writer) burgers_store_chain<false>(S, C, lane, c, R);
        __syncthreads();
    }
}

}  // namespace ipmcmc
