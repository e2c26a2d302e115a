// Metropolis machinery shared by the Burgers (chain per warp) and Lorenz (chain per lane group)
// kernels: proposal, accept/reject, Welford moments, counters, optional traces.
//
//   proposal   v = coef_u*u + coef_w*w        proposer.py:29-30 (RW: 1, sqrt(2 delta)),
//                                             proposer.py:81-82 (pCN: sqrt(1-beta^2), beta),
//                                             proposer.py:53-56,110-115 (VarStep: per-step table)
//   w          N(0,C) draw = factor @ z       distribution.py:114-118 (numpy svd map)
//   accept     a > U, a = exp(I(u)-I(v))      accepter.py:59-62 (strict, un-clipped, NaN rejects)
//              I = t*Phi (+ 0.5||L w||^2 RW)  accepter.py:98-106, 121-122; t = inverse temperature
//                                             (replica exchange, tempering.cuh), 1 for the reference
//   constraint reject before drawing U        accepter.py:52-55
//   counters   calls / accepts                accepter.py:13-36
//   recording  sampler.py:18-28 (burn-in max(0, b - si), thinning si)
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace ipmcmc {

struct SamplerDev {
    int d, proposer, accepter, factor_kind, recompute_phi_u, has_constraint;
    double coef_u, coef_w;
    const double *coef_sched;  // device [2*n_sched] or nullptr
    long long n_sched;
    const double *factor;      // device [d] or [d*d]
    const double *prior_chol;  // device [d*d]
    double box_lo[IPMCMC_MAX_DIM], box_hi[IPMCMC_MAX_DIM], box_shift[IPMCMC_MAX_DIM];
    // wide path (IPMCMC_MAX_DIM < d <= IPMCMC_MAX_DIM_WIDE): device tables instead of the arrays above
    const double *box_wide;         // [3*d] = lo | hi | shift, or nullptr
    const double *prior_chol_diag;  // [d] diagonal of the prior Cholesky factor (ACCEPT_RW), or nullptr
    unsigned long long seed;
    long long chain_offset, first_step, record_start, record_interval;
};

struct ChainBufDev {
    double *u, *phi, *model_state, *mom_count, *mom_mean, *mom_m2;
    long long *counters;
    double *trace;
    long long n_record;
    double *steplog, *vlog;
    const double *inject_w, *inject_u;
    const int *slot_chain;
    int n_slots;
    long long *sched;   // dynamic step scheduler scratch (int64 [3*n_chains + 2]) or nullptr
    const double *inv_temp;  // [n_chains] inverse temperature of each chain's likelihood, or nullptr (= 1)
};

enum : int { CNT_CALLS = 0, CNT_ACCEPTS, CNT_WORK_A, CNT_WORK_B, CNT_NONFINITE, CNT_CONSTRAINT, CNT_N };

// Lane-group view: a chain is served by `GL` consecutive lanes starting at `base` (GL = 32 for
// Burgers, K for Lorenz); component i of u lives on group lane i.
struct Group {
    int base, gl, lane;  // lane = index inside the group
    unsigned mask;
    __device__ __forceinline__ double bcast(double v, int src) const { return __shfl_sync(mask, v, base + src); }
};

__device__ __forceinline__ void step_coefs(const SamplerDev &S, long long gstep, double &a, double &b) {
    if (S.coef_sched) {
        const long long i = gstep < S.n_sched ? gstep : S.n_sched - 1;
        a = S.coef_sched[2 * i];
        b = S.coef_sched[2 * i + 1];
    } else {
        a = S.coef_u;
        b = S.coef_w;
    }
}

// Proposal noise w_i for component i = group lane (0 for lanes >= d).
__device__ __forceinline__ double proposal_noise(const SamplerDev &S, const ChainBufDev &C, const Group &G,
                                                 long long chain_local, long long chain_global, long long s,
                                                 long long n_steps, long long gstep) {
    const int i = G.lane;
    if (C.inject_w) return (i < S.d) ? C.inject_w[(chain_local * n_steps + s) * S.d + i] : 0.0;
    const double z = (i < S.d) ? draw_normal(S.seed, (uint64_t)chain_global, (uint64_t)gstep, (uint32_t)i) : 0.0;
    if (S.factor_kind == 0) return z;
    if (S.factor_kind == 1) return (i < S.d) ? S.factor[i] * z : 0.0;
    double w = 0.0;
    for (int j = 0; j < S.d; ++j) {
        const double zj = G.bcast(z, j);
        if (i < S.d) w = w + S.factor[i * S.d + j] * zj;
    }
    return w;
}

// 0.5 * ||L x||^2 as the reference evaluates it: .5 * np.linalg.norm(L @ x)**2 (accepter.py:104-106)
__device__ __forceinline__ double prior_regulariser(const SamplerDev &S, const Group &G, double x) {
    const int i = G.lane;
    double y = 0.0;
    for (int j = 0; j < S.d; ++j) {
        const double xj = G.bcast(x, j);
        if (i < S.d && j <= i) y = y + S.prior_chol[i * S.d + j] * xj;
    }
    double ss = 0.0;
    for (int j = 0; j < S.d; ++j) {
        const double yj = G.bcast(y, j);
        ss = ss + yj * yj;
    }
    const double nrm = sqrt(ss);
    return 0.5 * (nrm * nrm);
}

__device__ __forceinline__ bool constraint_ok(const SamplerDev &S, const Group &G, double v) {
    const int i = G.lane;
    bool ok = true;
    if (i < S.d) {
        const double s = v + S.box_shift[i];
        ok = (s > S.box_lo[i]) && (s < S.box_hi[i]);
    }
    // all lanes of the group must agree
    const unsigned bal = __ballot_sync(G.mask, ok);
    const unsigned gmask = (G.gl == 32) ? 0xffffffffu : (((1u << G.gl) - 1u) << G.base);
    return (bal & gmask) == gmask;
}

// Number of recorded steps in [record_start, g): recorded are the g with (g - record_start + 1) % interval == 0
// (sampler.py:23-28).
__device__ __forceinline__ long long recorded_before(const SamplerDev &S, long long g) {
    if (!(S.record_interval > 0 && g > S.record_start)) return 0;
    return (g - S.record_start) / S.record_interval;
}
__device__ __forceinline__ bool records_step(const SamplerDev &S, long long gstep) {
    if (!(S.record_interval > 0 && gstep >= S.record_start)) return false;
    return ((gstep - S.record_start + 1) % S.record_interval) == 0;
}

struct Welford {
    double count, mean, m2;
    __device__ __forceinline__ void add(double x) {
        count += 1.0;
        const double delta = x - mean;
        mean += delta / count;
        m2 += delta * (x - mean);
    }
};

}  // namespace ipmcmc
