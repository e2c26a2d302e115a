/*
 * ipmcmc.h -- C ABI of the B200-native batched MCMC engine (libipmcmc.so).
 *
 * The reference (ochsnerd/ip_mcmc) is pure Python and has NO FFI: its "plugin API" is a set of
 * duck-typed callables.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference root); ip_mcmc_b200/ binds them with ctypes and re-exposes
 * them under the reference's class names (see INTEGRATION.md for the binding stub).
 *
 * Conventions
 *   - every function returns 0 on success, a negative IPMCMC_E* code otherwise;
 *     ipmcmc_last_error() returns a thread-local message for the last failure.
 *   - "dev" pointers are CUDA device pointers owned by the CALLER (torch allocates them);
 *     "host" pointers are ordinary host memory.  The library never frees caller memory and
 *     owns only the small constant tables inside an ipmcmc_problem.
 *   - all work is enqueued on the cudaStream_t passed as `stream` (void*, may be NULL = legacy
 *     default stream) and is asynchronous unless the function name ends in _host.
 *   - all floating point is IEEE binary64.  Arrays are C-contiguous.
 *   - a handle is not thread-safe; use one per host thread / GPU.
 */
#ifndef IPMCMC_H
#define IPMCMC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IPMCMC_ABI_VERSION 2

#define IPMCMC_MAX_DIM 32   /* parameter dimension d held on the lanes of one warp (3 in every
                               reference script): every feature, dynamic scheduler, team solver    */
#define IPMCMC_MAX_DIM_WIDE 256 /* Burgers with a truncated KL prior of up to 253 modes: the parameter
                               vector lives in shared memory ("wide path"): N <= 1024 cells, diagonal
                               sampling factor (factor_kind 0/1), diagonal prior_chol, static scheduler */
#define IPMCMC_MAX_OBS 64   /* observation dimension q (5 Burgers, 5K = 30 Lorenz)            */

enum {
    IPMCMC_OK = 0,
    IPMCMC_EINVAL = -1,      /* bad argument (mirrors the reference's asserts)                 */
    IPMCMC_ECUDA = -2,       /* CUDA runtime error                                             */
    IPMCMC_EUNSUPPORTED = -3 /* configuration outside what the kernels are instantiated for    */
};

enum { IPMCMC_MODEL_BURGERS = 1, IPMCMC_MODEL_LORENZ = 2 };

/* numerics of the Burgers finite-volume update */
enum {
    IPMCMC_NUMERICS_EXACT = 0, /* the reference's floating-point operation order: bit-identical
                                  end states / G / Phi (no FMA contraction)                   */
    IPMCMC_NUMERICS_FUSED = 1  /* FMA-contracted update; agrees with EXACT to <= 3.4e-11 relative */
};

/* ipmcmc_burgers_desc.flags */
enum {
    IPMCMC_BURGERS_NO_MONOTONE_SHORTCUT = 1 /* FUSED numerics: always reduce max|u| over all cells for the CFL
                                               step instead of taking it from the two end cells of a monotone
                                               state (results are bit-identical; used by the tests to prove it) */
};

/* proposal / acceptance kinds */
enum { IPMCMC_PROPOSE_RW = 0, IPMCMC_PROPOSE_PCN = 1 };
enum { IPMCMC_ACCEPT_RW = 0, IPMCMC_ACCEPT_PCN = 1 };

typedef struct ipmcmc_problem ipmcmc_problem; /* opaque: forward model + potential constants   */

/* --------------------------------------------------------------------------------------------
 * Gaussian-misfit potential  Phi(u) = -logpdf_N(0,Sigma)(y - G(u))
 *   replaces EvolutionPotential.__call__            ip_mcmc/ip_mcmc/potential.py:53-54
 *   and GaussianDistribution.logpdf                 ip_mcmc/ip_mcmc/distribution.py:111-112
 * scipy evaluates it as 0.5*((rank*log(2pi) + log_pdet) + sum(square(dev @ LP))).
 * ------------------------------------------------------------------------------------------ */
typedef struct ipmcmc_potential_desc {
    int32_t n_obs;            /* q                                                              */
    int32_t whiten_dense;     /* 0: LP has one non-zero per column (diagonal Sigma, possibly
                                    permuted by eigh): r_i = dev[perm[i]] * scale[i]
                                 1: dense LP (row-major q x q), r_i = sum_j dev[j]*LP[j][i]      */
    const double *y;          /* host [q]   data                                                */
    const int32_t *perm;      /* host [q]   (whiten_dense == 0)                                 */
    const double *scale;      /* host [q]   (whiten_dense == 0)                                 */
    const double *LP;         /* host [q*q] (whiten_dense == 1)                                 */
    double log_const;         /* rank*log(2pi) + log_pdet                                       */
} ipmcmc_potential_desc;

/* --------------------------------------------------------------------------------------------
 * Burgers forward model  G(u) = Measurer(RusanovFVM.integrate(PerturbedRiemannIC(mean + u), T))
 *   replaces FVMObservationOperator.__call__        report/scripts/burgers/utilities.py:40-41
 *            PerturbedRiemannIC                     report/scripts/burgers/utilities.py:44-62
 *            RusanovMCMC / RusanovFVM               utilities.py:65-79, rusanov.py:15-109
 *            Measurer                               report/scripts/burgers/utilities.py:82-109
 * Grid tables (cell centres, dx, measurement windows) are computed on the host with NumPy exactly
 * as the reference does (linspace/searchsorted) and passed in.
 * ------------------------------------------------------------------------------------------ */
typedef struct ipmcmc_burgers_desc {
    int32_t n_cells;          /* N interior cells (the solver carries N+2 with ghosts)          */
    int32_t numerics;         /* IPMCMC_NUMERICS_*                                              */
    int32_t max_fv_steps;     /* safety cap on FV time steps per solve; <= 0: 8*N + 256.  A solve takes
                                 T*N*<max|u|> steps (dt = dx/2 / max|u|, domain length 2): the default
                                 admits states up to |u| ~ 8 (the reference's prior: 2.5 +- 0.25) and
                                 stops the blow-up solves the reference's interior-only CFL produces
                                 when the jump falls between a ghost and the first cell centre
                                 (rusanov.py:102-109; ~300 N steps there).  A capped solve reports
                                 Phi = NaN: rejected and counted (counters[4])                    */
    int32_t n_params;         /* d = 3 + n_kl_modes: (delta_1, delta_2, sigma, a_1..a_m)        */
    double T;                 /* end time (the last step is NOT clipped, rusanov.py:40-45)      */
    double dx;                /* solver spacing = linspace retstep (rusanov.py:22-25)           */
    double dx_meas;           /* Measurer spacing x[1]-x[0] (utilities.py:91)                   */
    const double *x;          /* host [N+2] cell centres incl. ghosts                           */
    const double *param_mean; /* host [d] prior mean added to u (utilities.py:41)               */
    const int32_t *win_left;  /* host [q] searchsorted limits into the interior array           */
    const int32_t *win_right; /* host [q]                                                       */
    /* Extension (not in the reference; BASELINE.json north_star "truncated KL/spectral prior"):
       w0(x) = PerturbedRiemannIC(x) + sum_k a_k * phi_k(x), the coefficients a_k being parameters
       3..3+m-1 with a diagonal (KL) prior.  kl_basis is phi_k at the N+2 cell centres.          */
    int32_t n_kl_modes;       /* m (0 = the reference's 3-parameter problem)                    */
    int32_t flags;            /* IPMCMC_BURGERS_* bits (0 = default)                            */
    const double *kl_basis;   /* host [m * (N+2)], row-major (mode, cell); NULL when m = 0      */
    ipmcmc_potential_desc potential;
} ipmcmc_burgers_desc;

/* --------------------------------------------------------------------------------------------
 * Lorenz-96 forward model  G(u) = time-mean of the 5K moment functions over one RK45 solve
 *   replaces LorenzObservationOperator.__call__     report/scripts/lorenz_mcmc.py:55-71
 *            Lorenz96.__call__                      report/scripts/lorenz.py:44-101
 *            moment_function                        report/scripts/lorenz_mcmc.py:17-40
 *            scipy.integrate.solve_ivp(RK45)        (third-party; call site lorenz_mcmc.py:70-71)
 * u = (F, h, b) perturbations of `param_mean`; c is fixed.  The initial condition is carried
 * from solve to solve per chain (lorenz_mcmc.py:66) in a caller-owned [n_chains, K*(J+1)] buffer.
 * ------------------------------------------------------------------------------------------ */
typedef struct ipmcmc_lorenz_desc {
    int32_t K, J;             /* slow variables (3 <= K <= IPMCMC_MAX_OBS/5 = 12) / fast variables per
                                 slow variable (J in {1,2,4,8})                                  */
    int32_t max_attempts;     /* cap on RK attempts per solve (<=0: 1<<20)                      */
    int32_t numerics;         /* IPMCMC_NUMERICS_EXACT: right-hand side in the reference's rounding
                                 order (lorenz.py:73-101); IPMCMC_NUMERICS_FUSED: contracted RHS  */
    double T;                 /* integration horizon per solve                                  */
    double c;                 /* fixed time-scale parameter                                     */
    double rtol, atol;        /* solve_ivp defaults 1e-3, 1e-6                                  */
    const double *param_mean; /* host [3] prior means of (F, h, b)                              */
    ipmcmc_potential_desc potential; /* n_obs must be 5*K                                       */
} ipmcmc_lorenz_desc;

int ipmcmc_burgers_create(const ipmcmc_burgers_desc *desc, ipmcmc_problem **out);
int ipmcmc_lorenz_create(const ipmcmc_lorenz_desc *desc, ipmcmc_problem **out);
void ipmcmc_destroy(ipmcmc_problem *p);

/* --------------------------------------------------------------------------------------------
 * Batched forward evaluation (no MCMC): G(u_c), Phi(u_c) for n independent parameter vectors.
 *   replaces observation_operator(u) and EvolutionPotential(u) called in a Python loop.
 * Optional outputs may be NULL.
 *   u_dev      [n, d]
 *   G_dev      [n, q]
 *   phi_dev    [n]
 *   state_dev  Burgers: [n, N] interior end state (RusanovMCMC.__call__, utilities.py:75-79)
 *              Lorenz : [n, K*(J+1)] IN: initial condition, OUT: state at t = T
 *   work_dev   [n, 2] int64: Burgers (FV time steps, 0); Lorenz (accepted, rejected RK attempts)
 * ------------------------------------------------------------------------------------------ */
int ipmcmc_forward(ipmcmc_problem *p, int64_t n, const double *u_dev, double *G_dev,
                   double *phi_dev, double *state_dev, int64_t *work_dev, void *stream);

/* --------------------------------------------------------------------------------------------
 * The fused Metropolis kernel: proposal -> forward model -> Phi -> accept/reject -> moments,
 * `n_steps` steps for `n_chains` independent chains in ONE launch.
 *   replaces MCMCSampler.run/_step                  ip_mcmc/ip_mcmc/sampler.py:12-41
 *            ConstStep/VarStep StandardRW / pCN proposers   proposer.py:14-115
 *            ProbabilisticAccepter / StandardRWAccepter / pCNAccepter  accepter.py:58-122
 *            ConstrainAccepter (box constraints)    accepter.py:39-55
 *            CountedAccepter                        accepter.py:13-36
 * ------------------------------------------------------------------------------------------ */
typedef struct ipmcmc_sampler_desc {
    int32_t dim;              /* d                                                              */
    int32_t proposer;         /* IPMCMC_PROPOSE_*                                               */
    int32_t accepter;         /* IPMCMC_ACCEPT_*                                                */
    int32_t factor_kind;      /* 0: w = z (identity), 1: w_i = factor[i]*z_i (diagonal),
                                 2: w = factor(d x d, row-major) @ z
                                 (GaussianDistribution.sample, distribution.py:114-118)         */
    int32_t recompute_phi_u;  /* 1: evaluate Phi(u) again every step before Phi(v), as the
                                 reference does (accepter.py:99-100,121-122); required for the
                                 stateful Lorenz operator, bit-equivalent to 0 for Burgers      */
    int32_t has_constraint;   /* 1: reject without drawing U when not lo < v+shift < hi         */
    int32_t reserved0, reserved1;
    /* v = coef_u * u + coef_w * w.  RW: (1, sqrt(2 delta)); pCN: (sqrt(1-beta^2), beta).
       If coef_sched_dev != NULL it is a device array [2 * n_sched] of (coef_u, coef_w) pairs
       indexed by the global step number (VarStep* proposers); steps >= n_sched use the last. */
    double coef_u, coef_w;
    const double *coef_sched_dev;
    int64_t n_sched;
    const double *factor;     /* host [d] or [d*d] per factor_kind (may be NULL for kind 0)     */
    const double *prior_chol; /* host [d*d] lower Cholesky factor L of the prior covariance,
                                 used by ACCEPT_RW: I(w) = Phi(w) + 0.5*||L w||^2
                                 (accepter.py:104-106; NOT the inverse -- accepter_test.py:29-30) */
    const double *box_lo;     /* host [d] (has_constraint)                                      */
    const double *box_hi;     /* host [d]                                                       */
    const double *box_shift;  /* host [d]                                                       */
    uint64_t seed;            /* Philox4x32-10 key = (seed lo, global chain id)                 */
    int64_t chain_offset;     /* global id of local chain 0 (multi-GPU sharding); global ids must
                                 stay below 2^32 (the Philox key holds 32 bits of it)           */
    int64_t first_step;       /* global index of the first step of this launch                  */
    int64_t record_start;     /* first step of the sampling phase = max(0, burn_in - interval)  */
    int64_t record_interval;  /* sample_interval (sampler.py:25-28); <=0: record nothing        */
} ipmcmc_sampler_desc;

typedef struct ipmcmc_chain_buffers {
    /* chain state, IN/OUT */
    double *u_dev;            /* [n_chains, d]                                                  */
    double *phi_dev;          /* [n_chains] Phi(u); NaN = not yet evaluated                     */
    double *model_state_dev;  /* Lorenz: [n_chains, K*(J+1)] carried IC; Burgers: NULL          */
    /* running posterior moments (Welford), IN/OUT */
    double *mom_count_dev;    /* [n_chains]                                                     */
    double *mom_mean_dev;     /* [n_chains, d]                                                  */
    double *mom_m2_dev;       /* [n_chains, d]                                                  */
    /* counters, IN/OUT: [n_chains, 6] int64 =
       (calls, accepts, forward work a, forward work b, non-finite Phi, constraint rejects)
       work a/b: Burgers (FV time steps, solves); Lorenz (accepted, rejected RK attempts)       */
    int64_t *counters_dev;
    /* optional OUT */
    double *trace_dev;        /* [n_chains, n_record, d] recorded samples of this launch        */
    int64_t n_record;         /* capacity of trace_dev per chain                                */
    double *steplog_dev;      /* [n_chains, n_steps, 4] = (Phi(v), a, accepted, forward work)   */
    double *vlog_dev;         /* [n_chains, n_steps, d] proposals                               */
    /* optional IN: injected noise (parity mode; the reference's MockRNG seam)                  */
    const double *inject_w_dev; /* [n_chains, n_steps, d] proposal normals at the w level       */
    const double *inject_u_dev; /* [n_chains, n_steps]    accept uniforms                       */
    /* reserved, ignored (formerly scheduling hints of a static chain -> warp map)                 */
    const void *reserved_ptr0;
    int32_t reserved0, reserved1;
    /* scratch of the DYNAMIC STEP SCHEDULER, the only path of Burgers chains with N <= 1024 and d <= 32
       (work unit: a chain) and of Lorenz chains (work unit: a warp's group of floor(32/K) chains): persistent
       warps take (unit, sched_chunk steps) work items from a FIFO of ready units, which keeps every SM
       sub-partition busy until the launch ends although solve lengths are data dependent.  Results do not
       depend on it.  int64 [sched_len >= 3*units + 2], contents irrelevant on entry; NULL: the library
       makes a stream-ordered allocation and frees it inside the call.  Ignored by the wide (d > 32) and
       team (N > 1024) Burgers paths.                                                               */
    int64_t *sched_dev;
    int64_t sched_len;
    int32_t sched_chunk;      /* Metropolis steps per work item (<= 0: Burgers min(4, max(1, n_steps/64)),
                                 Lorenz 1)                                                          */
    int32_t reserved;
} ipmcmc_chain_buffers;

int ipmcmc_run(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, const ipmcmc_chain_buffers *b,
               int64_t n_chains, int64_t n_steps, void *stream);

/* --------------------------------------------------------------------------------------------
 * Replica exchange (parallel tempering) for Burgers chains.  Not in the reference.
 * A tempered batch is n_ladders x K chains, ladder-major: local chain c = l*K + k is rung k of ladder l
 * (global id chain_offset + c; chain_offset a multiple of K, so a shard owns whole ladders).
 *
 * ipmcmc_run_tempered: ipmcmc_run with the likelihood of chain c tempered by inv_temp_dev[c] (t, [n_chains]):
 *   a = exp((t*Phi(u) + reg_u) - (t*Phi(v) + reg_v)),  accepted = a > U
 * reg is the RW regulariser 0.5*||L w||^2 (0 for pCN) and is not tempered; Phi itself stays untempered in
 * phi_dev and the step log.  t = 1 gives ipmcmc_run's results bit for bit.  Lorenz chains: IPMCMC_EUNSUPPORTED
 * (their Phi depends on the carried initial condition).
 * ------------------------------------------------------------------------------------------ */
int ipmcmc_run_tempered(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, const ipmcmc_chain_buffers *b,
                        const double *inv_temp_dev, int64_t n_chains, int64_t n_steps, void *stream);
/* One swap round r (>= 0) between adjacent rungs, run after global step (r+1)*swap_interval.  It proposes the
 * pairs (k, k+1) with k = r (mod 2) in every ladder and swaps iff
 *   exp((t_k - t_{k+1}) * (Phi_k - Phi_{k+1})) > U      (strict; NaN never swaps)
 * U = Philox4x32-10 keyed (seed lo, global id of slot k), counter (r lo, r hi, 0xFFFFFFFE, seed hi) -- a slot
 * no Metropolis draw uses -- or inject_u_dev[l*(K-1) + k] when inject_u_dev [n_ladders, K-1] is not NULL.
 * On a swap the rows of u_dev [n_ladders*K, dim], the entries of phi_dev and the rows of replica_dev move;
 * Welford moments, counters and traces stay with the slot.
 *   replica_dev      [n_ladders*K, 2] int32 (replica id, direction); start from (k, 0).  After the swaps slot 0
 *                    gets direction +1, incrementing round_trips_dev[l] if it was -1, and slot K-1 gets -1
 *                    (in the rounds that propose pair (0,1), resp. pair (K-2,K-1)).
 *   swap_counts_dev  [n_ladders, K-1, 2] int64 (attempts, accepts) per adjacent pair, accumulated
 *   round_trips_dev  [n_ladders] int64, accumulated
 * Arguments are checked before any CUDA call: K >= 2, n_ladders >= 1, 1 <= dim <= 256, round >= 0,
 * chain_offset % K == 0, global ids below 2^32, and every pointer but inject_u_dev non-NULL. */
int ipmcmc_swap_replicas(int64_t n_ladders, int32_t ladder_size, int32_t dim, double *u_dev, double *phi_dev,
                         const double *inv_temp_dev, uint64_t seed, int64_t chain_offset, int64_t round,
                         const double *inject_u_dev, int32_t *replica_dev, int64_t *swap_counts_dev,
                         int64_t *round_trips_dev, void *stream);

/* Pool per-chain Welford moments and counters of n_chains chains into
 *   pooled_dev[0] = n, [1..d] = mean, [1+d..2d] = M2, then the 6 counters as doubles
 * (2d + 7 doubles) with Chan's parallel merge as a fixed tree (deterministic; two small launches whose
 * cost does not grow with n_chains beyond reading 8(1+2d)+48 bytes per chain) -- the buffer each rank
 * contributes to the ONE collective of a multi-GPU run (ip_mcmc_b200/parallel.py).
 *   replaces the post-hoc np.mean / np.var over sample arrays and CountedAccepter.ratio()
 *   (burgers_mcmc.py:136-143, accepter.py:29-36) for batches whose samples are not materialised.
 * scratch_dev: caller-owned device scratch of ipmcmc_pool_scratch_bytes(n_chains, dim) bytes, or NULL
 * (then a stream-ordered allocation is made and freed inside the call). */
int64_t ipmcmc_pool_scratch_bytes(int64_t n_chains, int32_t dim);
int ipmcmc_pool_moments(int64_t n_chains, int32_t dim, const double *mom_count_dev,
                        const double *mom_mean_dev, const double *mom_m2_dev,
                        const int64_t *counters_dev, double *pooled_dev, void *scratch_dev,
                        int64_t scratch_bytes, void *stream);

/* --------------------------------------------------------------------------------------------
 * Convergence diagnostics of a recorded trace, computed on the device for every chain of a batch.
 *   replaces stats.integrated_autocorr_time / stats.ess_multichain called per chain on the host, and adds
 *   split-R-hat (BDA3 section 11.4) and multi-chain ESS (BDA3 section 11.5); the estimators are restated
 *   in NumPy in ip_mcmc_b200/stats.py (integrated_autocorr_time, split_rhat, multichain_ess).
 * The trace is [n_chains, n_draws, dim] as ipmcmc_run writes it, with rows contiguous and chains
 * `chain_stride` >= n_draws*dim doubles apart (a view trace[:, burn:] needs no copy).  The split
 * estimators use the first and the last h = n_draws/2 draws of each chain as m = 2*n_chains sequences
 * (n_draws >= 4).  Every result is deterministic: its summation order depends on (n_chains, n_draws, dim)
 * only, not on the device, the launch geometry or whether scratch is supplied.
 * scratch_dev: caller-owned device scratch of ipmcmc_diag_scratch_bytes(n_chains, dim, n_lags) bytes (n_lags
 * the largest lag block the caller asks for; 0 for seqstats only), or NULL: a stream-ordered allocation is
 * made and freed inside the call.
 * ------------------------------------------------------------------------------------------ */
int64_t ipmcmc_diag_scratch_bytes(int64_t n_chains, int32_t dim, int64_t n_lags);
/* Per-chain integrated autocorrelation time with Geyer's initial-positive-sequence cut-off
 * (stats.integrated_autocorr_time): tau_dev [n_chains, dim].  A constant series gives
 * 1 + 4*floor((n_draws-1)/2), as the host's all-ones autocorrelation does.  One warp per series. */
int ipmcmc_diag_tau(int64_t n_chains, int64_t n_draws, int32_t dim, const double *trace_dev,
                    int64_t chain_stride, double *tau_dev, void *stream);
/* Split-sequence statistics per parameter j (BDA3 section 11.4): seqstats_dev [dim, 4] =
 * (m, mean of the sequence means, M2 = sum of squared deviations of the sequence means, sum of the
 * sequence variances s_s^2 with ddof = 1).  Rows of several batches merge with Chan's formula
 * (ip_mcmc_b200/parallel.py:merge_seqstats). */
int ipmcmc_diag_seqstats(int64_t n_chains, int64_t n_draws, int32_t dim, const double *trace_dev,
                         int64_t chain_stride, double *seqstats_dev, void *scratch_dev,
                         int64_t scratch_bytes, void *stream);
/* Variogram sums (BDA3 section 11.5) for the lags t in [lag0, lag0 + n_lags), lag0 + n_lags <= h:
 *   vsum_dev[j*vsum_ld + (t - lag0)] = sum_s sum_{i=t}^{h-1} (psi_{s,i} - psi_{s,i-t})^2
 * over the split sequences psi_s.  Parameters with done_dev[j] != 0 are skipped (their row is not
 * written); done_dev may be NULL.  Sums of several batches add. */
int ipmcmc_diag_variogram(int64_t n_chains, int64_t n_draws, int32_t dim, const double *trace_dev,
                          int64_t chain_stride, int64_t lag0, int64_t n_lags, const int32_t *done_dev,
                          double *vsum_dev, int64_t vsum_ld, void *scratch_dev, int64_t scratch_bytes,
                          void *stream);
/* Truncated autocorrelation sum and final estimates from seqstats_dev [dim, 4] and the variogram sums
 * vsum_dev[j*vsum_ld + t] of the lags 1 <= t < lag_end (lag_end <= h); called after each block of lags
 * with a growing lag_end, the last call with lag_end = h.  rho_t = 1 - V_t/(2 var+), V_t = vsum_t/(m(h-t)),
 * var+ = (h-1)/h W + B/h, W = sum s_s^2/m, B = h/(m-1) M2.  With S = 0, t = 1:
 *   S += rho_t; stop if t+2 > h-1 or rho_{t+1} + rho_{t+2} < 0; else S += rho_{t+1}, t += 2, repeat.
 * state_dev [2*dim] (zero before the first call) carries the loop between calls, which pauses where a
 * lag it needs is not summed yet; done_dev [dim] int32 (zero before the first call) is set when a
 * parameter's loop ends, and then out_dev [3*dim] = (R-hat = sqrt(var+/W), n_eff = m h/(1 + 2S), T = t)
 * for it.  IEEE arithmetic throughout: all sequences constant give NaN, constant ones at different
 * values inf. */
int ipmcmc_diag_truncate(int64_t n_draws, int32_t dim, const double *seqstats_dev, const double *vsum_dev,
                         int64_t vsum_ld, int64_t lag_end, double *state_dev, int32_t *done_dev,
                         double *out_dev, void *stream);

/* --------------------------------------------------------------------------------------------
 * Host-buffer entry point -- what a non-Python binding of MCMCSampler.run (sampler.py:12-33) calls, and
 * what bench.py times as `e2e_c_abi`: copies u0 (and the Lorenz IC) host->device, runs n_steps with the
 * SAME kernels and scheduler as the device-buffer path (dynamic step scheduler where it applies), copies
 * the recorded samples, final states, per-chain counters and pooled moments device->host, synchronises.
 * All device memory is one stream-ordered arena allocated and freed inside the call.
 * ------------------------------------------------------------------------------------------ */
typedef struct ipmcmc_host_io {
    const double *u0_host;     /* IN  [n_chains, d] initial states                                  */
    const double *phi0_host;   /* IN  [n_chains] Phi(u0) from a previous call (phi_host), or NULL:
                                      the kernel evaluates it (one extra solve per chain)           */
    double *model_state_host;  /* IN/OUT Lorenz [n_chains, K*(J+1)] carried IC; Burgers NULL        */
    double *samples_host;      /* OUT [n_chains, n_record, d] recorded samples, or NULL             */
    int64_t n_record;          /*     capacity per chain of samples_host                            */
    double *u_host;            /* OUT [n_chains, d] final states, or NULL                           */
    double *phi_host;          /* OUT [n_chains] Phi(final state), or NULL                          */
    int64_t *counters_host;    /* OUT [n_chains, 6], or NULL                                        */
    double *pooled_host;       /* OUT [2d + 7] pooled moments + counters, or NULL                   */
    int32_t reserved;          /* ignored (formerly the choice of a static scheduler)               */
    int32_t sched_chunk;       /* Metropolis steps per work item (<= 0: Burgers min(4, max(1, n_steps/64)), Lorenz 1) */
} ipmcmc_host_io;

int ipmcmc_sample_host(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, int64_t n_chains,
                       int64_t n_steps, const ipmcmc_host_io *io, void *stream);

/* --------------------------------------------------------------------------------------------
 * d-dimensional histogram of recorded samples, ACCUMULATED into hist_dev across calls -- the device half of
 *   np.histogramdd(chain.T, bins=n_bins, range=intervals)   report/scripts/burgers/burgers_wasserstein_chain.py:182-184,
 *                                                           burgers_wasserstein_grid.py:205-231
 * so that a 100 000-step study keeps bins^d counters instead of its samples.
 *   samples_dev [n, stride] (the first `dim` entries of each row are used; a trace of ipmcmc_run is [., d])
 *   shift_dev   [dim] added to every sample first (the scripts add the prior mean, chain.py:257-259)
 *   edges_dev   [dim, bins+1] bin edges per dimension (np.linspace(lo, hi, bins+1)); numpy semantics:
 *               right-open bins, the last edge belongs to the last bin, outside values are dropped
 *   hist_dev    [bins^dim] int64 counters, row-major over dimensions, updated with atomic adds
 * ------------------------------------------------------------------------------------------ */
int ipmcmc_histogram_accumulate(int64_t n, int32_t dim, int32_t bins, const double *samples_dev,
                                int64_t stride, const double *shift_dev, const double *edges_dev,
                                int64_t *hist_dev, void *stream);

/* --------------------------------------------------------------------------------------------
 * Probes used by the parity tests and the roofline measurement
 * ------------------------------------------------------------------------------------------ */
/* Lorenz-96 RHS for n states (lorenz.py:44-101): theta_dev [n,4] = (F,h,c,b). */
int ipmcmc_lorenz_rhs(int32_t K, int32_t J, int32_t numerics, int64_t n, const double *theta_dev,
                      const double *state_dev, double *rhs_dev, void *stream);
/* One Dormand-Prince attempt (scipy rk.py:14-72,111-116) for n states with step h_dev[n]:
   out_dev [n, 2*n_var + 1] = (y_new, f_new, error_norm). */
int ipmcmc_lorenz_rk45_attempt(int32_t K, int32_t J, int32_t numerics, int64_t n, const double *theta_dev,
                               const double *state_dev, const double *h_dev, double rtol,
                               double atol, double *out_dev, void *stream);
/* Engine RNG: out_dev [n_chains, n_steps, d + 1] = (normals xi_0..xi_{d-1}, uniform U). */
int ipmcmc_rng_probe(uint64_t seed, int64_t chain_offset, int64_t first_step, int64_t n_chains,
                     int64_t n_steps, int32_t dim, double *out_dev, void *stream);
/* The branch-free IEEE division of the EXACT positive-monotone Burgers loop (dt = (dx/2) / max|u|, rusanov.py:102-109)
   beside the compiler's:  q_fast_dev[i] = div_rn_fast(a, b_dev[i]),  q_ieee_dev[i] = a / b_dev[i]  (must be the same
   bits for 1e-100 < b < 1e100). */
int ipmcmc_div_probe(int64_t n, double a, const double *b_dev, double *q_fast_dev, double *q_ieee_dev, void *stream);
/* Dependent-free DFMA micro-benchmark: returns measured fp64 FMA throughput in TFLOP/s
   (2 flops per FMA) of the current device, timed with CUDA events over `iters` launches.  */
int ipmcmc_fp64_peak(int32_t iters, double *tflops_out);

const char *ipmcmc_last_error(void);
int ipmcmc_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* IPMCMC_H */
