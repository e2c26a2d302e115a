// libipmcmc.so -- C ABI (include/ipmcmc.h) over the sm_100a kernels.  This unit holds the ABI, the Lorenz
// kernels and the small kernels; the Burgers kernels are compiled from burgers_inst.cu, one unit per
// cells-per-lane value.  Build (ip_mcmc_b200/build.py): nvcc -gencode arch=compute_100a,code=sm_100a -O3
// -lineinfo -fmad=false -c <unit> ..., then nvcc -shared.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "burgers_launch.cuh"
#include "diag.cuh"
#include "lorenz_kernels.cuh"
#include "tempering.cuh"

using namespace ipmcmc;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) return fail(IPMCMC_ECUDA, "%s: %s", #expr, cudaGetErrorString(_e));  \
    } while (0)

extern "C" const char *ipmcmc_last_error(void) { return g_err.c_str(); }
extern "C" int ipmcmc_abi_version(void) { return IPMCMC_ABI_VERSION; }

// ------------------------------------------------------------------------------------------------
// problem handle
// ------------------------------------------------------------------------------------------------
struct ipmcmc_problem {
    int model = 0;
    int numerics = 0;
    BurgersDev b;
    LorenzDev l;
    std::vector<void *> owned;   // device allocations freed in destroy
    // Small sampler tables (proposal factor, prior Cholesky factor) by content: a table is uploaded once,
    // synchronously, and never overwritten, so launches on different streams or with different samplers
    // cannot race on it and repeated launches do not re-upload it.
    struct Table {
        std::vector<double> host;
        double *dev;
    };
    std::vector<Table> tables;
};

static int cached_table(ipmcmc_problem *p, const double *host, size_t n, const double **dev) {
    for (const auto &t : p->tables)
        if (t.host.size() == n && memcmp(t.host.data(), host, n * sizeof(double)) == 0) {
            *dev = t.dev;
            return 0;
        }
    if (p->tables.size() >= 64) return fail(IPMCMC_EUNSUPPORTED, "more than 64 distinct sampler tables on one problem handle");
    double *d = nullptr;
    CUDA_TRY(cudaMalloc((void **)&d, n * sizeof(double)));
    p->owned.push_back(d);
    CUDA_TRY(cudaMemcpy(d, host, n * sizeof(double), cudaMemcpyHostToDevice));
    p->tables.push_back(ipmcmc_problem::Table{std::vector<double>(host, host + n), d});
    *dev = d;
    return 0;
}

static int upload(ipmcmc_problem *p, const void *host, size_t bytes, void **dev) {
    CUDA_TRY(cudaMalloc(dev, bytes ? bytes : 8));
    p->owned.push_back(*dev);
    if (bytes) CUDA_TRY(cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice));
    return 0;
}

static int fill_potential(ipmcmc_problem *p, const ipmcmc_potential_desc &d, PotentialDev &out) {
    if (d.n_obs < 1 || d.n_obs > IPMCMC_MAX_OBS) return fail(IPMCMC_EINVAL, "n_obs=%d outside [1,%d]", d.n_obs, IPMCMC_MAX_OBS);
    if (!d.y) return fail(IPMCMC_EINVAL, "potential.y is NULL");
    memset(&out, 0, sizeof out);
    out.q = d.n_obs;
    out.dense = d.whiten_dense ? 1 : 0;
    out.log_const = d.log_const;
    for (int i = 0; i < d.n_obs; ++i) out.y[i] = d.y[i];
    if (!out.dense) {
        if (!d.perm || !d.scale) return fail(IPMCMC_EINVAL, "potential.perm/scale is NULL");
        for (int i = 0; i < d.n_obs; ++i) {
            if (d.perm[i] < 0 || d.perm[i] >= d.n_obs) return fail(IPMCMC_EINVAL, "potential.perm[%d] out of range", i);
            out.perm[i] = d.perm[i];
            out.scale[i] = d.scale[i];
        }
    } else {
        if (!d.LP) return fail(IPMCMC_EINVAL, "potential.LP is NULL");
        void *dev;
        int rc = upload(p, d.LP, sizeof(double) * d.n_obs * d.n_obs, &dev);
        if (rc) return rc;
        out.LP = (const double *)dev;
    }
    return 0;
}

static int finish_create(ipmcmc_problem *p, ipmcmc_problem **out) {
    *out = p;
    return 0;
}

extern "C" void ipmcmc_destroy(ipmcmc_problem *p) {
    if (!p) return;
    for (void *d : p->owned) cudaFree(d);
    delete p;
}

static const int kCPL[] = {1, 2, 4, 7, 8, 16, 32};

static int pick_cpl(int N) {
    for (int c : kCPL)
        if (32 * c >= N) return c;
    return 0;
}

extern "C" int ipmcmc_burgers_create(const ipmcmc_burgers_desc *d, ipmcmc_problem **out) {
    if (!d || !out) return fail(IPMCMC_EINVAL, "NULL argument");
    if (d->n_cells < 2) return fail(IPMCMC_EINVAL, "n_cells=%d < 2", d->n_cells);
    if (!pick_cpl(d->n_cells) && d->n_cells != 2048 && d->n_cells != 4096)
        return fail(IPMCMC_EUNSUPPORTED, "n_cells=%d: grids above 1024 cells must be 2048 or 4096 (2 or 4 warps per chain)", d->n_cells);
    if (d->n_kl_modes < 0 || d->n_kl_modes > IPMCMC_MAX_DIM_WIDE - 3) return fail(IPMCMC_EUNSUPPORTED, "n_kl_modes=%d outside [0,%d]", d->n_kl_modes, IPMCMC_MAX_DIM_WIDE - 3);
    if (d->n_params > IPMCMC_MAX_DIM && d->n_cells > 1024)
        return fail(IPMCMC_EUNSUPPORTED, "more than %d parameters (wide path) need n_cells <= 1024", IPMCMC_MAX_DIM);
    if (d->n_params != 3 + d->n_kl_modes) return fail(IPMCMC_EINVAL, "n_params=%d, expected 3 + n_kl_modes = %d", d->n_params, 3 + d->n_kl_modes);
    if (d->n_kl_modes > 0 && !d->kl_basis) return fail(IPMCMC_EINVAL, "kl_basis is NULL");
    if (d->numerics != IPMCMC_NUMERICS_EXACT && d->numerics != IPMCMC_NUMERICS_FUSED) return fail(IPMCMC_EINVAL, "bad numerics");
    if (!d->x || !d->param_mean || !d->win_left || !d->win_right) return fail(IPMCMC_EINVAL, "NULL table");
    if (!(d->dx > 0)) return fail(IPMCMC_EINVAL, "dx must be > 0");
    auto *p = new ipmcmc_problem();
    p->model = IPMCMC_MODEL_BURGERS;
    p->numerics = d->numerics;
    BurgersDev &b = p->b;
    memset(&b, 0, sizeof b);
    b.N = d->n_cells;
    b.d = d->n_params;
    b.max_fv_steps = d->max_fv_steps > 0 ? d->max_fv_steps : 8 * d->n_cells + 256;   // include/ipmcmc.h: max_fv_steps
    b.T = d->T;
    b.dx = d->dx;
    b.half_dx = 0.5 * d->dx;
    b.neg_inv_dx = -1.0 / d->dx;
    int ex;
    b.dx_pow2 = (std::frexp(d->dx, &ex) == 0.5) ? 1 : 0;
    b.dx_meas = d->dx_meas;
    b.no_mono = (d->flags & IPMCMC_BURGERS_NO_MONOTONE_SHORTCUT) ? 1 : 0;
    for (int i = 0; i < b.d && i < IPMCMC_MAX_DIM; ++i) b.param_mean[i] = d->param_mean[i];
    int rc = 0;
    if (b.d > IPMCMC_MAX_DIM) {   // wide path: the means as a device table
        void *pm;
        rc = upload(p, d->param_mean, sizeof(double) * b.d, &pm);
        if (rc) { ipmcmc_destroy(p); return rc; }
        b.param_mean_wide = (const double *)pm;
    }
    rc = fill_potential(p, d->potential, b.pot);
    if (rc) { ipmcmc_destroy(p); return rc; }
    for (int i = 0; i < b.pot.q; ++i) {
        const int l = d->win_left[i], r = d->win_right[i];
        if (l < 0 || r > b.N || l > r) { ipmcmc_destroy(p); return fail(IPMCMC_EINVAL, "window %d = [%d,%d) outside [0,%d]", i, l, r, b.N); }
        b.win_left[i] = l;
        b.win_right[i] = r;
    }
    void *dev;
    rc = upload(p, d->x, sizeof(double) * (b.N + 2), &dev);
    if (rc) { ipmcmc_destroy(p); return rc; }
    b.x = (const double *)dev;
    b.n_modes = d->n_kl_modes;
    if (b.n_modes > 0) {
        rc = upload(p, d->kl_basis, sizeof(double) * (size_t)b.n_modes * (b.N + 2), &dev);
        if (rc) { ipmcmc_destroy(p); return rc; }
        b.basis = (const double *)dev;
    }
    rc = finish_create(p, out);
    if (rc) ipmcmc_destroy(p);
    return rc;
}

extern "C" int ipmcmc_lorenz_create(const ipmcmc_lorenz_desc *d, ipmcmc_problem **out) {
    if (!d || !out) return fail(IPMCMC_EINVAL, "NULL argument");
    if (d->K < 3 || 5 * d->K > IPMCMC_MAX_OBS)
        return fail(IPMCMC_EUNSUPPORTED, "K=%d outside [3,%d] (one lane per slow variable; 5K observations <= IPMCMC_MAX_OBS)", d->K, IPMCMC_MAX_OBS / 5);
    if (d->J != 1 && d->J != 2 && d->J != 4 && d->J != 8) return fail(IPMCMC_EUNSUPPORTED, "J=%d not in {1,2,4,8}", d->J);
    if (d->potential.n_obs != 5 * d->K) return fail(IPMCMC_EINVAL, "n_obs=%d, expected 5*K=%d", d->potential.n_obs, 5 * d->K);
    if (!d->param_mean) return fail(IPMCMC_EINVAL, "NULL param_mean");
    auto *p = new ipmcmc_problem();
    p->model = IPMCMC_MODEL_LORENZ;
    LorenzDev &l = p->l;
    memset(&l, 0, sizeof l);
    l.K = d->K;
    l.J = d->J;
    l.nvar = d->K * (d->J + 1);
    l.max_attempts = d->max_attempts > 0 ? d->max_attempts : (1 << 20);
    if (d->numerics != IPMCMC_NUMERICS_EXACT && d->numerics != IPMCMC_NUMERICS_FUSED) {
        delete p;
        return fail(IPMCMC_EINVAL, "bad numerics");
    }
    p->numerics = d->numerics;
    l.T = d->T;
    l.c = d->c;
    l.rtol = d->rtol;
    l.atol = d->atol;
    for (int i = 0; i < 3; ++i) l.param_mean[i] = d->param_mean[i];
    int rc = fill_potential(p, d->potential, l.pot);
    if (rc) { ipmcmc_destroy(p); return rc; }
    rc = finish_create(p, out);
    if (rc) ipmcmc_destroy(p);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// dispatch
// ------------------------------------------------------------------------------------------------
static int cu(cudaError_t e) {
    if (e != cudaSuccess) return fail(IPMCMC_ECUDA, "kernel launch: %s", cudaGetErrorString(e));
    return 0;
}

// runs body(scratch) on the caller's scratch (checked against need) or a stream-ordered allocation
template <class F>
static int with_scratch(void *scratch, int64_t scratch_bytes, int64_t need, cudaStream_t st, const F &body) {
    if (scratch) {
        if (scratch_bytes < need) return fail(IPMCMC_EINVAL, "scratch: %lld bytes given, %lld needed", (long long)scratch_bytes, (long long)need);
        return body(scratch);
    }
    void *tmp = nullptr;
    CUDA_TRY(cudaMallocAsync(&tmp, (size_t)need, st));
    const int rc = body(tmp);
    cudaFreeAsync(tmp, st);
    return rc;
}

#define BURGERS_TEAM_DISPATCH(FN, ...)                                                                  \
    do {                                                                                                \
        const bool fused = p->numerics == IPMCMC_NUMERICS_FUSED;                                        \
        if (p->b.N == 2048) return cu(fused ? FN<NUM_FUSED, 2>(__VA_ARGS__) : FN<NUM_EXACT, 2>(__VA_ARGS__)); \
        if (p->b.N == 4096) return cu(fused ? FN<NUM_FUSED, 4>(__VA_ARGS__) : FN<NUM_EXACT, 4>(__VA_ARGS__)); \
    } while (0)

#define BURGERS_CASE(FN, C, ...)                                                                        \
    case C:                                                                                             \
        if (fused) return cu(padded ? FN<C, NUM_FUSED, true>(__VA_ARGS__) : FN<C, NUM_FUSED, false>(__VA_ARGS__)); \
        return cu(padded ? FN<C, NUM_EXACT, true>(__VA_ARGS__) : FN<C, NUM_EXACT, false>(__VA_ARGS__));

#define BURGERS_DISPATCH(FN, ...)                                                       \
    do {                                                                                \
        const int cpl = pick_cpl(p->b.N);                                               \
        const bool fused = p->numerics == IPMCMC_NUMERICS_FUSED;                        \
        const bool padded = p->b.N != 32 * cpl;                                         \
        switch (cpl) {                                                                  \
            BURGERS_CASE(FN, 1, __VA_ARGS__)                                            \
            BURGERS_CASE(FN, 2, __VA_ARGS__)                                            \
            BURGERS_CASE(FN, 4, __VA_ARGS__)                                            \
            BURGERS_CASE(FN, 7, __VA_ARGS__)                                            \
            BURGERS_CASE(FN, 8, __VA_ARGS__)                                            \
            BURGERS_CASE(FN, 16, __VA_ARGS__)                                           \
            BURGERS_CASE(FN, 32, __VA_ARGS__)                                           \
        }                                                                               \
        return fail(IPMCMC_EUNSUPPORTED, "no kernel for n_cells=%d", p->b.N);           \
    } while (0)

// CTA shape of the Lorenz kernels.  Batches that fit one wave get one CTA of W = ceil(warps / n_SM)
// warps per SM, so that the warps of an SM are dealt round-robin onto its four sub-partitions
// (warp w -> sub-partition w % 4); larger batches use 4-warp CTAs and the block scheduler.
static int lorenz_cta_warps(long long warps, int K) {
    int n_sm = 148;
    sm_count(n_sm);
    int wpc = warps <= 8LL * n_sm ? (int)((warps + n_sm - 1) / n_sm) : 4;
    if (const char *e = getenv("IPMCMC_LORENZ_WPC")) wpc = atoi(e) > 0 && atoi(e) <= 8 ? atoi(e) : wpc;  // experiments
    if (wpc > lorenz_warps_fit(K)) wpc = lorenz_warps_fit(K);
    return wpc < 1 ? 1 : wpc;
}

// J in {1,2,4,8}; K = 6 (the reference's problem) is specialised at compile time, any other K
// runs the generic lane-group code; NUM = IPMCMC_NUMERICS_*.
#define LORENZ_DISPATCH_JK(KERNEL, J, KT, NUM, ...)                                     \
    do {                                                                                \
        if ((NUM) == IPMCMC_NUMERICS_FUSED) KERNEL<J, KT, LNUM_FUSED> __VA_ARGS__;      \
        else KERNEL<J, KT, LNUM_EXACT> __VA_ARGS__;                                     \
    } while (0)
#define LORENZ_DISPATCH(KERNEL, J, K, NUM, ...)                                         \
    do {                                                                                \
        if ((NUM) != IPMCMC_NUMERICS_EXACT && (NUM) != IPMCMC_NUMERICS_FUSED)           \
            return fail(IPMCMC_EINVAL, "bad numerics");                                 \
        switch (J) {                                                                    \
            case 1: LORENZ_DISPATCH_JK(KERNEL, 1, 0, NUM, __VA_ARGS__); break;          \
            case 2: LORENZ_DISPATCH_JK(KERNEL, 2, 0, NUM, __VA_ARGS__); break;          \
            case 4:                                                                     \
                if ((K) == 6) LORENZ_DISPATCH_JK(KERNEL, 4, 6, NUM, __VA_ARGS__);       \
                else LORENZ_DISPATCH_JK(KERNEL, 4, 0, NUM, __VA_ARGS__);                \
                break;                                                                  \
            case 8: LORENZ_DISPATCH_JK(KERNEL, 8, 0, NUM, __VA_ARGS__); break;          \
            default: return fail(IPMCMC_EUNSUPPORTED, "J=%d not in {1,2,4,8}", J);      \
        }                                                                               \
        CUDA_TRY(cudaGetLastError());                                                   \
    } while (0)

extern "C" int ipmcmc_forward(ipmcmc_problem *p, int64_t n, const double *u_dev, double *G_dev, double *phi_dev,
                              double *state_dev, int64_t *work_dev, void *stream) {
    if (!p || !u_dev) return fail(IPMCMC_EINVAL, "NULL argument");
    if (n <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (p->model == IPMCMC_MODEL_BURGERS) {
        if (p->b.N > 1024)
            BURGERS_TEAM_DISPATCH(burgers_launch_team_forward, p->b, n, u_dev, G_dev, phi_dev, state_dev, (long long *)work_dev, st);
        if (p->b.d > IPMCMC_MAX_DIM)
            BURGERS_DISPATCH(burgers_launch_wide_forward, p->b, n, u_dev, G_dev, phi_dev, state_dev, (long long *)work_dev, st);
        BURGERS_DISPATCH(burgers_launch_forward, p->b, n, u_dev, G_dev, phi_dev, state_dev, (long long *)work_dev, st);
    }
    if (!state_dev) return fail(IPMCMC_EINVAL, "Lorenz forward needs state_dev (carried initial condition)");
    const int groups = lorenz_groups(p->l.K);
    const long long warps = (n + groups - 1) / groups;
    const int wpc = lorenz_cta_warps(warps, p->l.K);
    LORENZ_DISPATCH(lorenz_forward_kernel, p->l.J, p->l.K, p->numerics,
                    <<<grid_for((warps + wpc - 1) / wpc), 32 * wpc, wpc * lorenz_smem_bytes(p->l.K), st>>>(
                        p->l, n, u_dev, G_dev, phi_dev, state_dev, (long long *)work_dev));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// sampler
// ------------------------------------------------------------------------------------------------
static int make_sampler(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, SamplerDev &S, int64_t n_chains) {
    const int d = s->dim;
    if (d < 1 || d > IPMCMC_MAX_DIM_WIDE) return fail(IPMCMC_EINVAL, "dim=%d outside [1,%d]", d, IPMCMC_MAX_DIM_WIDE);
    if (p->model == IPMCMC_MODEL_BURGERS && d != p->b.d) return fail(IPMCMC_EINVAL, "dim=%d but the forward model takes %d parameters", d, p->b.d);
    const bool wide = d > IPMCMC_MAX_DIM;
    if (wide && s->factor_kind == 2) return fail(IPMCMC_EUNSUPPORTED, "dim=%d > %d: the wide path samples with a diagonal factor only", d, IPMCMC_MAX_DIM);
    if (p->model == IPMCMC_MODEL_LORENZ && d != 3) return fail(IPMCMC_EINVAL, "dim=%d but the Lorenz operator takes (F,h,b)", d);
    if (s->proposer != IPMCMC_PROPOSE_RW && s->proposer != IPMCMC_PROPOSE_PCN) return fail(IPMCMC_EINVAL, "bad proposer");
    if (s->accepter != IPMCMC_ACCEPT_RW && s->accepter != IPMCMC_ACCEPT_PCN) return fail(IPMCMC_EINVAL, "bad accepter");
    if (s->factor_kind < 0 || s->factor_kind > 2) return fail(IPMCMC_EINVAL, "bad factor_kind");
    if (s->factor_kind && !s->factor) return fail(IPMCMC_EINVAL, "factor is NULL");
    if (s->accepter == IPMCMC_ACCEPT_RW && !s->prior_chol) return fail(IPMCMC_EINVAL, "ACCEPT_RW needs prior_chol");
    if (s->coef_sched_dev && s->n_sched < 1) return fail(IPMCMC_EINVAL, "empty schedule");
    // Philox is keyed by the low 32 bits of the global chain id (philox.cuh)
    if (s->chain_offset < 0 || s->chain_offset + n_chains > (1LL << 32))
        return fail(IPMCMC_EUNSUPPORTED, "global chain ids must lie in [0, 2^32): chain_offset=%lld n_chains=%lld",
                    (long long)s->chain_offset, (long long)n_chains);
    memset(&S, 0, sizeof S);
    S.d = d;
    S.proposer = s->proposer;
    S.accepter = s->accepter;
    S.factor_kind = s->factor_kind;
    S.recompute_phi_u = s->recompute_phi_u;
    S.has_constraint = s->has_constraint;
    S.coef_u = s->coef_u;
    S.coef_w = s->coef_w;
    S.coef_sched = s->coef_sched_dev;
    S.n_sched = s->n_sched;
    if (s->factor_kind) {
        int rc = cached_table(p, s->factor, s->factor_kind == 1 ? (size_t)d : (size_t)d * d, &S.factor);
        if (rc) return rc;
    }
    if (s->accepter == IPMCMC_ACCEPT_RW && !wide) {
        int rc = cached_table(p, s->prior_chol, (size_t)d * d, &S.prior_chol);
        if (rc) return rc;
    }
    if (s->accepter == IPMCMC_ACCEPT_RW && wide) {   // diagonal prior factor only
        std::vector<double> diag(d);
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) {
                if (i == j) diag[i] = s->prior_chol[(size_t)i * d + j];
                else if (s->prior_chol[(size_t)i * d + j] != 0.0)
                    return fail(IPMCMC_EUNSUPPORTED, "dim=%d > %d: the wide path needs a diagonal prior_chol", d, IPMCMC_MAX_DIM);
            }
        int rc = cached_table(p, diag.data(), (size_t)d, &S.prior_chol_diag);
        if (rc) return rc;
    }
    if (s->has_constraint && wide) {
        if (!s->box_lo || !s->box_hi) return fail(IPMCMC_EINVAL, "constraint box is NULL");
        std::vector<double> box(3 * (size_t)d);
        for (int i = 0; i < d; ++i) {
            box[i] = s->box_lo[i];
            box[d + i] = s->box_hi[i];
            box[2 * d + i] = s->box_shift ? s->box_shift[i] : 0.0;
        }
        int rc = cached_table(p, box.data(), box.size(), &S.box_wide);
        if (rc) return rc;
    }
    if (s->has_constraint && !wide) {
        if (!s->box_lo || !s->box_hi) return fail(IPMCMC_EINVAL, "constraint box is NULL");
        for (int i = 0; i < d; ++i) {
            S.box_lo[i] = s->box_lo[i];
            S.box_hi[i] = s->box_hi[i];
            S.box_shift[i] = s->box_shift ? s->box_shift[i] : 0.0;
        }
    }
    S.seed = s->seed;
    S.chain_offset = s->chain_offset;
    S.first_step = s->first_step;
    S.record_start = s->record_start;
    S.record_interval = s->record_interval;
    return 0;
}

// ipmcmc_run (inv_temp NULL) and ipmcmc_run_tempered
static int run_chains(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, const ipmcmc_chain_buffers *b,
                      const double *inv_temp, int64_t n_chains, int64_t n_steps, void *stream) {
    if (!p || !s || !b) return fail(IPMCMC_EINVAL, "NULL argument");
    if (inv_temp && p->model == IPMCMC_MODEL_LORENZ)
        return fail(IPMCMC_EUNSUPPORTED, "Lorenz chains cannot be tempered: Phi(u) depends on the carried initial "
                                         "condition, so a replica swap is not a valid Metropolis move for them");
    if (n_chains <= 0 || n_steps < 0) return fail(IPMCMC_EINVAL, "n_chains=%lld n_steps=%lld", (long long)n_chains, (long long)n_steps);
    if (!b->u_dev || !b->phi_dev || !b->mom_count_dev || !b->mom_mean_dev || !b->mom_m2_dev || !b->counters_dev)
        return fail(IPMCMC_EINVAL, "chain state buffer is NULL");
    if (p->model == IPMCMC_MODEL_LORENZ && !b->model_state_dev) return fail(IPMCMC_EINVAL, "Lorenz chains need model_state_dev");
    cudaStream_t st = (cudaStream_t)stream;
    SamplerDev S;
    int rc = make_sampler(p, s, S, n_chains);
    if (rc) return rc;
    ChainBufDev C;
    C.u = b->u_dev;
    C.phi = b->phi_dev;
    C.model_state = b->model_state_dev;
    C.mom_count = b->mom_count_dev;
    C.mom_mean = b->mom_mean_dev;
    C.mom_m2 = b->mom_m2_dev;
    C.counters = (long long *)b->counters_dev;
    C.trace = b->trace_dev;
    C.n_record = b->n_record;
    C.steplog = b->steplog_dev;
    C.vlog = b->vlog_dev;
    C.inject_w = b->inject_w_dev;
    C.inject_u = b->inject_u_dev;
    C.inv_temp = inv_temp;
    if (p->model == IPMCMC_MODEL_BURGERS) {
        if (p->b.N > 1024) BURGERS_TEAM_DISPATCH(burgers_launch_team_chain, p->b, S, C, n_chains, n_steps, st);
        if (S.d > IPMCMC_MAX_DIM) BURGERS_DISPATCH(burgers_launch_wide_chain, p->b, S, C, n_chains, n_steps, st);
        if (n_chains >= (1LL << 31)) return fail(IPMCMC_EUNSUPPORTED, "dynamic scheduler: n_chains >= 2^31");
    }
    // Every other chain runs on the dynamic step scheduler (sched.cuh), whose work unit is a Burgers chain or a warp's
    // group of Lorenz chains.  Metropolis steps per work item: an item costs ~4 us of queue traffic and state reloads,
    // so long Burgers launches use longer items (measured on B200, 1024 x 256 cells: +1 % at 200 steps per launch; 50
    // steps: none).  A Lorenz item is two RK45 solves of a warp's chain group (~1.7 ms): one step per item balances best
    // (4096 chains, 128 steps per launch: 1.87 M chain-steps/s against 1.83 M with two steps per item).
    const bool lorenz = p->model == IPMCMC_MODEL_LORENZ;
    const int groups = lorenz ? lorenz_groups(p->l.K) : 1;
    const long long units = (n_chains + groups - 1) / groups;
    int chunk = b->sched_chunk > 0 ? b->sched_chunk : lorenz ? 1 : (int)(n_steps / 64 < 1 ? 1 : (n_steps / 64 > 4 ? 4 : n_steps / 64));
    if (const char *e = getenv("IPMCMC_SCHED_CHUNK")) chunk = atoi(e) > 0 ? atoi(e) : chunk;  // experiments
    const int64_t sched_bytes = b->sched_dev ? b->sched_len * (int64_t)sizeof(int64_t) : 0;
    return with_scratch(b->sched_dev, sched_bytes, sched_len(units) * (int64_t)sizeof(int64_t), st, [&](void *sched) {
        C.sched = (long long *)sched;
        if (!lorenz) BURGERS_DISPATCH(burgers_launch_chain_queue, p->b, S, C, n_chains, n_steps, chunk, st);
        // Lorenz: persistent warps, one wave (255 registers: 8 warps per SM at most; the queue needs every launched CTA resident)
        const long long warps = units;   // one warp per chain group
        const int wpc = lorenz_cta_warps(warps, p->l.K);
        int n_sm = 148;
        CUDA_TRY(sm_count(n_sm));
        long long ctas;
        int qwpc = wpc;
        if (warps <= 8LL * n_sm) {
            // one wave: one CTA per SM, ceil(warps / n_SM) warps each -- every SM gets work (820 groups at 4096
            // chains: 80 SMs with 6 warps, 68 with 5, instead of 137 CTAs of 6 and 11 idle SMs)
            ctas = warps < n_sm ? warps : n_sm;
            qwpc = (int)((warps + ctas - 1) / ctas);
            const int fit = lorenz_warps_fit(p->l.K);
            if (qwpc > fit) { qwpc = fit; ctas = (warps + qwpc - 1) / qwpc; }
        } else {
            const long long resident = (long long)n_sm * (8 / wpc);
            ctas = (warps + wpc - 1) / wpc;
            if (ctas > resident) ctas = resident;
        }
        CUDA_TRY(sched_init(C.sched, warps, st));
        LORENZ_DISPATCH(lorenz_chain_queue_kernel, p->l.J, p->l.K, p->numerics,
                        <<<(int)ctas, 32 * qwpc, qwpc * lorenz_smem_bytes(p->l.K), st>>>(p->l, S, C, n_chains, n_steps, chunk));
        return 0;
    });
}

extern "C" int ipmcmc_run(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, const ipmcmc_chain_buffers *b,
                          int64_t n_chains, int64_t n_steps, void *stream) {
    return run_chains(p, s, b, nullptr, n_chains, n_steps, stream);
}

extern "C" int ipmcmc_run_tempered(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, const ipmcmc_chain_buffers *b,
                                   const double *inv_temp_dev, int64_t n_chains, int64_t n_steps, void *stream) {
    if (!inv_temp_dev) return fail(IPMCMC_EINVAL, "inv_temp_dev is NULL (use ipmcmc_run for untempered chains)");
    return run_chains(p, s, b, inv_temp_dev, n_chains, n_steps, stream);
}

// ------------------------------------------------------------------------------------------------
// replica exchange (tempering.cuh)
// ------------------------------------------------------------------------------------------------
extern "C" int ipmcmc_swap_replicas(int64_t n_ladders, int32_t ladder_size, int32_t dim, double *u_dev, double *phi_dev,
                                    const double *inv_temp_dev, uint64_t seed, int64_t chain_offset, int64_t round,
                                    const double *inject_u_dev, int32_t *replica_dev, int64_t *swap_counts_dev,
                                    int64_t *round_trips_dev, void *stream) {
    const int K = ladder_size;
    if (K < 2 || n_ladders < 1) return fail(IPMCMC_EINVAL, "ladder_size=%d (at least 2) n_ladders=%lld (at least 1)", K, (long long)n_ladders);
    if (dim < 1 || dim > IPMCMC_MAX_DIM_WIDE) return fail(IPMCMC_EINVAL, "dim=%d outside [1,%d]", dim, IPMCMC_MAX_DIM_WIDE);
    if (round < 0) return fail(IPMCMC_EINVAL, "round=%lld < 0", (long long)round);
    if (chain_offset < 0 || chain_offset % K != 0)
        return fail(IPMCMC_EINVAL, "chain_offset=%lld is not a multiple of ladder_size=%d: a ladder would be split", (long long)chain_offset, K);
    if (n_ladders > ((1LL << 32) - chain_offset) / K)
        return fail(IPMCMC_EUNSUPPORTED, "global chain ids must lie in [0, 2^32): chain_offset=%lld n_ladders=%lld ladder_size=%d",
                    (long long)chain_offset, (long long)n_ladders, K);
    if (!u_dev || !phi_dev || !inv_temp_dev || !replica_dev || !swap_counts_dev || !round_trips_dev)
        return fail(IPMCMC_EINVAL, "NULL argument");
    SwapDev W;
    W.n_ladders = n_ladders;
    W.chain_offset = chain_offset;
    W.round = round;
    W.K = K;
    W.d = dim;
    W.parity = (int)(round & 1);
    W.n_pairs = (K - W.parity) / 2;
    W.seed = seed;
    W.u = u_dev;
    W.phi = phi_dev;
    W.inv_temp = inv_temp_dev;
    W.inject_u = inject_u_dev;
    W.replica = replica_dev;
    W.swap_counts = (long long *)swap_counts_dev;
    W.round_trips = (long long *)round_trips_dev;
    if (W.n_pairs == 0) return 0;   // K = 2, odd round: no pair
    const long long warps = n_ladders * W.n_pairs;
    swap_round_kernel<<<grid_for((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(W);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// pooling of per-chain moments: Chan et al. merge as a fixed tree (deterministic: the tree depends on
// n_chains only, not on the launch geometry or the SM count)
//   pass 1: CTA b reduces chains [b*POOL_CHUNK, (b+1)*POOL_CHUNK); blockIdx.y = component j < d, or
//           d + k for counter k.  Thread t merges its chains t, t+256, ... in order, then the 256 partial
//           triples are merged by a shuffle-xor tree inside each warp and a sequential pass over the
//           8 warps -> partial[b][j] = (n, mean_j, M2_j)   (counters: exact int64 sums)
//   pass 2: one CTA, thread j merges partial[0..n_blocks)[j] in block order.
// 65 536 chains: 32 CTAs x (d + 6) rows, a few microseconds (the former single-thread-per-component loop
// took 0.35 ms per 1024 chains).
// ------------------------------------------------------------------------------------------------
constexpr int POOL_THREADS = 256;
constexpr int POOL_CHUNK = 2048;

__global__ void __launch_bounds__(POOL_THREADS) pool_partial_kernel(long long n_chains, int d,
                                                                    const double *__restrict__ cnt,
                                                                    const double *__restrict__ mean,
                                                                    const double *__restrict__ m2,
                                                                    const long long *__restrict__ counters,
                                                                    double *__restrict__ partial_mom,      // [n_blocks, d, 3]
                                                                    long long *__restrict__ partial_cnt) { // [n_blocks, CNT_N]
    __shared__ Mom3 smom[POOL_THREADS / 32];
    __shared__ long long scnt[POOL_THREADS / 32];
    const int t = threadIdx.x, j = blockIdx.y, lane = t & 31, warp = t >> 5;
    const long long c0 = (long long)blockIdx.x * POOL_CHUNK;
    const long long c1 = c0 + POOL_CHUNK < n_chains ? c0 + POOL_CHUNK : n_chains;
    if (j < d) {
        Mom3 acc{0.0, 0.0, 0.0};
        for (long long c = c0 + t; c < c1; c += POOL_THREADS) {
            const double nb = cnt[c];
            if (nb > 0.0) acc = chan_merge(acc, Mom3{nb, mean[c * d + j], m2[c * d + j]});
        }
#pragma unroll
        for (int off = 1; off < 32; off *= 2) {
            Mom3 o{__shfl_xor_sync(FULL, acc.n, off), __shfl_xor_sync(FULL, acc.mean, off), __shfl_xor_sync(FULL, acc.m2, off)};
            acc = (lane & off) ? chan_merge(o, acc) : chan_merge(acc, o);   // lower lane first: same bits on both
        }
        if (lane == 0) smom[warp] = acc;
        __syncthreads();
        if (t == 0) {
            Mom3 r = smom[0];
            for (int w = 1; w < POOL_THREADS / 32; ++w) r = chan_merge(r, smom[w]);
            double *o = partial_mom + ((long long)blockIdx.x * d + j) * 3;
            o[0] = r.n;
            o[1] = r.mean;
            o[2] = r.m2;
        }
    } else {
        const int k = j - d;
        long long sum = 0;
        for (long long c = c0 + t; c < c1; c += POOL_THREADS) sum += counters[c * CNT_N + k];
#pragma unroll
        for (int off = 16; off > 0; off /= 2) sum += __shfl_xor_sync(FULL, sum, off);
        if (lane == 0) scnt[warp] = sum;
        __syncthreads();
        if (t == 0) {
            long long r = 0;
            for (int w = 0; w < POOL_THREADS / 32; ++w) r += scnt[w];
            partial_cnt[(long long)blockIdx.x * CNT_N + k] = r;
        }
    }
}

__global__ void __launch_bounds__(64) pool_final_kernel(int n_blocks, int d, const double *__restrict__ partial_mom,
                                                        const long long *__restrict__ partial_cnt,
                                                        double *__restrict__ out) {
    for (int j = threadIdx.x; j < d + CNT_N; j += blockDim.x) {
        if (j < d) {
            Mom3 r{0.0, 0.0, 0.0};
            for (int b = 0; b < n_blocks; ++b) {
                const double *p = partial_mom + ((long long)b * d + j) * 3;
                r = chan_merge(r, Mom3{p[0], p[1], p[2]});
            }
            out[1 + j] = r.mean;
            out[1 + d + j] = r.m2;
            if (j == 0) out[0] = r.n;
        } else {
            long long sum = 0;
            for (int b = 0; b < n_blocks; ++b) sum += partial_cnt[(long long)b * CNT_N + (j - d)];
            out[1 + 2 * d + (j - d)] = (double)sum;
        }
    }
}

extern "C" int64_t ipmcmc_pool_scratch_bytes(int64_t n_chains, int32_t dim) {
    const long long nb = (n_chains + POOL_CHUNK - 1) / POOL_CHUNK;
    return (int64_t)(nb * (3LL * dim * sizeof(double) + CNT_N * sizeof(long long)));
}

static int pool_launch(long long n_chains, int d, const double *cnt, const double *mean, const double *m2,
                       const long long *counters, double *pooled, void *scratch, cudaStream_t st) {
    const long long nb = (n_chains + POOL_CHUNK - 1) / POOL_CHUNK;
    if (nb > 65535LL * 1024) return fail(IPMCMC_EUNSUPPORTED, "n_chains=%lld too large to pool", n_chains);
    double *pmom = (double *)scratch;
    long long *pcnt = (long long *)(pmom + nb * 3 * d);
    pool_partial_kernel<<<dim3((unsigned)nb, (unsigned)(d + CNT_N)), POOL_THREADS, 0, st>>>(n_chains, d, cnt, mean, m2, counters, pmom, pcnt);
    CUDA_TRY(cudaGetLastError());
    pool_final_kernel<<<1, 64, 0, st>>>((int)nb, d, pmom, pcnt, pooled);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int ipmcmc_pool_moments(int64_t n_chains, int32_t dim, const double *mom_count_dev,
                                   const double *mom_mean_dev, const double *mom_m2_dev, const int64_t *counters_dev,
                                   double *pooled_dev, void *scratch_dev, int64_t scratch_bytes, void *stream) {
    if (dim < 1 || dim > IPMCMC_MAX_DIM_WIDE) return fail(IPMCMC_EINVAL, "dim=%d", dim);
    if (n_chains < 1) return fail(IPMCMC_EINVAL, "n_chains=%lld", (long long)n_chains);
    if (!mom_count_dev || !mom_mean_dev || !mom_m2_dev || !counters_dev || !pooled_dev) return fail(IPMCMC_EINVAL, "NULL argument");
    const int64_t need = ipmcmc_pool_scratch_bytes(n_chains, dim);
    cudaStream_t st = (cudaStream_t)stream;
    if (scratch_dev) {
        if (scratch_bytes < need) return fail(IPMCMC_EINVAL, "pool scratch: %lld bytes given, %lld needed", (long long)scratch_bytes, (long long)need);
        return pool_launch(n_chains, dim, mom_count_dev, mom_mean_dev, mom_m2_dev, (const long long *)counters_dev, pooled_dev, scratch_dev, st);
    }
    void *tmp = nullptr;   // no caller scratch: stream-ordered allocation
    CUDA_TRY(cudaMallocAsync(&tmp, (size_t)need, st));
    const int rc = pool_launch(n_chains, dim, mom_count_dev, mom_mean_dev, mom_m2_dev, (const long long *)counters_dev, pooled_dev, tmp, st);
    cudaFreeAsync(tmp, st);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// convergence diagnostics of a recorded trace (diag.cuh)
// ------------------------------------------------------------------------------------------------
static int diag_check(int64_t n_chains, int64_t n, int32_t dim, const double *trace, int64_t stride, int64_t n_min) {
    if (n_chains < 1) return fail(IPMCMC_EINVAL, "n_chains=%lld", (long long)n_chains);
    if (n < n_min) return fail(IPMCMC_EINVAL, "n_draws=%lld (at least %lld)", (long long)n, (long long)n_min);
    if (n > 2147483647LL) return fail(IPMCMC_EUNSUPPORTED, "n_draws=%lld (at most 2^31 - 1)", (long long)n);
    if (dim < 1 || dim > IPMCMC_MAX_DIM_WIDE) return fail(IPMCMC_EINVAL, "dim=%d", dim);
    if (stride < n * dim) return fail(IPMCMC_EINVAL, "chain_stride=%lld < n_draws*dim=%lld", (long long)stride, (long long)(n * dim));
    if (!trace) return fail(IPMCMC_EINVAL, "NULL trace");
    return 0;
}

static long long seq_blocks(long long M) { return (M + SEQ_CHUNK - 1) / SEQ_CHUNK; }
static long long vario_blocks(long long M) { const long long c = vario_chunk(M); return (M + c - 1) / c; }

extern "C" int64_t ipmcmc_diag_scratch_bytes(int64_t n_chains, int32_t dim, int64_t n_lags) {
    if (n_chains < 1 || dim < 1 || n_lags < 0) return 0;
    const long long a = seq_blocks(n_chains) * dim * 4, b = vario_blocks(n_chains) * dim * n_lags;
    return (int64_t)((a > b ? a : b) * sizeof(double));
}

extern "C" int ipmcmc_diag_tau(int64_t n_chains, int64_t n_draws, int32_t dim, const double *trace_dev, int64_t chain_stride,
                               double *tau_dev, void *stream) {
    if (int rc = diag_check(n_chains, n_draws, dim, trace_dev, chain_stride, 1)) return rc;
    if (!tau_dev) return fail(IPMCMC_EINVAL, "NULL tau_dev");
    const long long series_bytes = n_draws * (long long)sizeof(double);
    const bool staged = series_bytes <= DIAG_SMEM;
    const int warps = staged ? (int)(DIAG_SMEM / series_bytes < 8 ? DIAG_SMEM / series_bytes : 8) : 8;
    const size_t smem = staged ? (size_t)(warps * series_bytes) : 0;
    const unsigned grid = (unsigned)grid_for((n_chains * dim + warps - 1) / warps);
    cudaStream_t st = (cudaStream_t)stream;
    if (staged) {
        CUDA_TRY(cudaFuncSetAttribute(diag_tau_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_SMEM));
        diag_tau_kernel<true><<<grid, 32 * warps, smem, st>>>(n_chains, n_draws, dim, trace_dev, chain_stride, tau_dev);
    } else {
        diag_tau_kernel<false><<<grid, 32 * warps, 0, st>>>(n_chains, n_draws, dim, trace_dev, chain_stride, tau_dev);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int ipmcmc_diag_seqstats(int64_t n_chains, int64_t n_draws, int32_t dim, const double *trace_dev,
                                    int64_t chain_stride, double *seqstats_dev, void *scratch_dev, int64_t scratch_bytes,
                                    void *stream) {
    if (int rc = diag_check(n_chains, n_draws, dim, trace_dev, chain_stride, 4)) return rc;
    if (!seqstats_dev) return fail(IPMCMC_EINVAL, "NULL seqstats_dev");
    const long long nb = seq_blocks(n_chains);
    if (nb > 2147483647LL) return fail(IPMCMC_EUNSUPPORTED, "n_chains=%lld", (long long)n_chains);
    cudaStream_t st = (cudaStream_t)stream;
    return with_scratch(scratch_dev, scratch_bytes, (int64_t)(nb * dim * 4 * sizeof(double)), st, [&](void *s) {
        double *part = (double *)s;
        diag_seq_partial_kernel<<<dim3((unsigned)nb, (unsigned)dim), DIAG_WARPS * 32, 0, st>>>(n_chains, n_draws, dim, trace_dev,
                                                                                              chain_stride, part);
        CUDA_TRY(cudaGetLastError());
        diag_seq_final_kernel<<<1, 64, 0, st>>>((int)nb, dim, part, seqstats_dev);
        CUDA_TRY(cudaGetLastError());
        return 0;
    });
}

extern "C" int ipmcmc_diag_variogram(int64_t n_chains, int64_t n_draws, int32_t dim, const double *trace_dev,
                                     int64_t chain_stride, int64_t lag0, int64_t n_lags, const int32_t *done_dev,
                                     double *vsum_dev, int64_t vsum_ld, void *scratch_dev, int64_t scratch_bytes, void *stream) {
    if (int rc = diag_check(n_chains, n_draws, dim, trace_dev, chain_stride, 4)) return rc;
    const long long h = n_draws / 2;
    if (lag0 < 0 || n_lags < 1 || lag0 + n_lags > h)
        return fail(IPMCMC_EINVAL, "lags [%lld, %lld) outside [0, h=%lld)", (long long)lag0, (long long)(lag0 + n_lags), h);
    if (!vsum_dev || vsum_ld < n_lags) return fail(IPMCMC_EINVAL, "vsum_dev=%p vsum_ld=%lld", (void *)vsum_dev, (long long)vsum_ld);
    const long long groups = (n_lags + 31) / 32;
    if (groups > 65535) return fail(IPMCMC_EUNSUPPORTED, "n_lags=%lld (at most %d per call)", (long long)n_lags, 65535 * 32);
    const long long nb = vario_blocks(n_chains);
    const bool staged = (long long)DIAG_WARPS * h * (long long)sizeof(double) <= DIAG_SMEM;
    cudaStream_t st = (cudaStream_t)stream;
    return with_scratch(scratch_dev, scratch_bytes, (int64_t)(nb * dim * n_lags * sizeof(double)), st, [&](void *s) {
        double *part = (double *)s;
        const dim3 grid((unsigned)nb, (unsigned)groups, (unsigned)dim);
        if (staged) {
            CUDA_TRY(cudaFuncSetAttribute(diag_vario_partial_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_SMEM));
            diag_vario_partial_kernel<true><<<grid, DIAG_WARPS * 32, (size_t)(DIAG_WARPS * h * sizeof(double)), st>>>(
                n_chains, n_draws, dim, trace_dev, chain_stride, lag0, n_lags, done_dev, part);
        } else {
            diag_vario_partial_kernel<false><<<grid, DIAG_WARPS * 32, 0, st>>>(n_chains, n_draws, dim, trace_dev, chain_stride,
                                                                              lag0, n_lags, done_dev, part);
        }
        CUDA_TRY(cudaGetLastError());
        const long long fb = (n_lags + 127) / 128;
        diag_vario_final_kernel<<<dim3((unsigned)(fb < 1024 ? fb : 1024), (unsigned)dim), 128, 0, st>>>((int)nb, dim, n_lags, part,
                                                                                                     done_dev, vsum_dev, vsum_ld);
        CUDA_TRY(cudaGetLastError());
        return 0;
    });
}

extern "C" int ipmcmc_diag_truncate(int64_t n_draws, int32_t dim, const double *seqstats_dev, const double *vsum_dev,
                                    int64_t vsum_ld, int64_t lag_end, double *state_dev, int32_t *done_dev, double *out_dev,
                                    void *stream) {
    const long long h = n_draws / 2;
    if (n_draws < 4 || dim < 1 || dim > IPMCMC_MAX_DIM_WIDE) return fail(IPMCMC_EINVAL, "n_draws=%lld dim=%d", (long long)n_draws, dim);
    if (lag_end < 1 || lag_end > h || vsum_ld < lag_end)
        return fail(IPMCMC_EINVAL, "lag_end=%lld vsum_ld=%lld (h=%lld)", (long long)lag_end, (long long)vsum_ld, h);
    if (!seqstats_dev || !vsum_dev || !state_dev || !done_dev || !out_dev) return fail(IPMCMC_EINVAL, "NULL argument");
    diag_truncate_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(h, dim, seqstats_dev, vsum_dev, vsum_ld, lag_end, state_dev,
                                                             done_dev, out_dev);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// d-dimensional histogram of recorded samples, accumulated across launches (chain-length / grid studies)
// ------------------------------------------------------------------------------------------------
// np.histogramdd semantics (numpy/lib/_histograms_impl.py): bin = searchsorted(edges, x, 'right') - 1 per
// dimension, a value on the last edge belongs to the last bin, values outside [first, last edge] are dropped.
// `edges` are the caller's (np.linspace) edges, so that the bin of a value on an edge is numpy's.
__global__ void __launch_bounds__(256) histogram_kernel(long long n, int d, int bins, const double *__restrict__ x,
                                                        long long stride, const double *__restrict__ shift,
                                                        const double *__restrict__ edges,
                                                        unsigned long long *__restrict__ hist) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        long long flat = 0;
        bool inside = true;
        for (int j = 0; j < d; ++j) {
            const double *e = edges + (long long)j * (bins + 1);
            const double v = x[i * stride + j] + shift[j];
            if (!(v >= e[0] && v <= e[bins])) {   // NaN is dropped too
                inside = false;
                break;
            }
            int k = (int)((v - e[0]) / (e[bins] - e[0]) * bins);
            k = k < 0 ? 0 : (k > bins - 1 ? bins - 1 : k);
            while (k > 0 && v < e[k]) --k;                      // exact searchsorted on the given edges
            while (k < bins - 1 && v >= e[k + 1]) ++k;
            flat = flat * bins + k;
        }
        if (inside) atomicAdd(hist + flat, 1ull);
    }
}

extern "C" int ipmcmc_histogram_accumulate(int64_t n, int32_t dim, int32_t bins, const double *samples_dev,
                                           int64_t stride, const double *shift_dev, const double *edges_dev,
                                           int64_t *hist_dev, void *stream) {
    if (dim < 1 || dim > IPMCMC_MAX_DIM || bins < 1) return fail(IPMCMC_EINVAL, "dim=%d bins=%d", dim, bins);
    if (n < 0 || stride < dim) return fail(IPMCMC_EINVAL, "n=%lld stride=%lld", (long long)n, (long long)stride);
    if (!samples_dev || !shift_dev || !edges_dev || !hist_dev) return fail(IPMCMC_EINVAL, "NULL argument");
    if (n == 0) return 0;
    const long long blocks = (n + 255) / 256;
    histogram_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, (cudaStream_t)stream>>>(
        n, dim, bins, samples_dev, stride, shift_dev, edges_dev, (unsigned long long *)hist_dev);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// host-buffer path
// ------------------------------------------------------------------------------------------------
__global__ void fill_kernel(double *p, long long n, double v) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}

static bool uses_queue(const ipmcmc_problem *p) {
    return p->model == IPMCMC_MODEL_LORENZ || (p->b.N <= 1024 && p->b.d <= IPMCMC_MAX_DIM);
}

// The arena of ipmcmc_sample_host comes from a pool of the library's own (one per device) that keeps its memory
// between calls: with the default pool's release threshold of zero every call paid the physical allocation of the
// whole arena again (tens of milliseconds for a 25 MB sample buffer, and the reason the C entry point's end-to-end
// figure varied from run to run).
static cudaMemPool_t arena_pool() {
    static cudaMemPool_t pools[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!pools[dev]) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        cudaMemPool_t mp = nullptr;
        if (cudaMemPoolCreate(&mp, &props) != cudaSuccess) return nullptr;
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
        pools[dev] = mp;
    }
    return pools[dev];
}

extern "C" int ipmcmc_sample_host(ipmcmc_problem *p, const ipmcmc_sampler_desc *s, int64_t n_chains, int64_t n_steps,
                                  const ipmcmc_host_io *io, void *stream) {
    if (!p || !s || !io || !io->u0_host) return fail(IPMCMC_EINVAL, "NULL argument");
    if (n_chains <= 0 || n_steps < 0) return fail(IPMCMC_EINVAL, "n_chains=%lld n_steps=%lld", (long long)n_chains, (long long)n_steps);
    const int d = s->dim;
    const int d_model = p->model == IPMCMC_MODEL_LORENZ ? 3 : p->b.d;
    if (d < 1 || d > IPMCMC_MAX_DIM_WIDE || d != d_model) return fail(IPMCMC_EINVAL, "dim=%d but the forward model takes %d parameters", d, d_model);
    if (io->n_record < 0) return fail(IPMCMC_EINVAL, "n_record=%lld", (long long)io->n_record);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)n_chains;
    const size_t nvar = p->model == IPMCMC_MODEL_LORENZ ? (size_t)p->l.nvar : 0;
    if (nvar && !io->model_state_host) return fail(IPMCMC_EINVAL, "Lorenz needs model_state_host");
    // one device arena: u | phi | count | mean | m2 | pooled | model_state | trace | counters | sched | pool scratch
    const size_t n_trace = io->samples_host ? B * (size_t)io->n_record * d : 0;
    const size_t n_dbl = B * d + B + B + B * d + B * d + (2 * d + 7) + B * nvar + n_trace;
    const size_t units = p->model == IPMCMC_MODEL_LORENZ ? (B + lorenz_groups(p->l.K) - 1) / lorenz_groups(p->l.K) : B;
    const size_t n_sched = uses_queue(p) ? (size_t)sched_len((long long)units) : 0;
    const size_t pool_bytes = (size_t)ipmcmc_pool_scratch_bytes(n_chains, d);
    double *arena = nullptr;
    cudaMemPool_t mem_pool = arena_pool();
    if (!mem_pool) return fail(IPMCMC_ECUDA, "cannot create the arena memory pool");
    CUDA_TRY(cudaMallocFromPoolAsync((void **)&arena, n_dbl * sizeof(double) + (B * CNT_N + n_sched) * sizeof(long long) + pool_bytes,
                                     mem_pool, st));
    double *u = arena, *phi = u + B * d, *cnt = phi + B, *mean = cnt + B, *m2 = mean + B * d, *pooled = m2 + B * d;
    double *mstate = pooled + (2 * d + 7), *trace = mstate + B * nvar;
    long long *counters = (long long *)(trace + n_trace), *sched = counters + B * CNT_N;
    void *pool_scratch = (void *)(sched + n_sched);
    int rc = 0;
    auto cleanup = [&](int code) {
        cudaFreeAsync(arena, st);
        return code;
    };
    cudaError_t e;
    e = cudaMemcpyAsync(u, io->u0_host, B * d * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && nvar) e = cudaMemcpyAsync(mstate, io->model_state_host, B * nvar * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(cnt, 0, (B + 2 * B * d) * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(counters, 0, B * CNT_N * sizeof(long long), st);
    if (e == cudaSuccess) {
        if (io->phi0_host) {   // Phi(u_0) known from a previous call: no extra solve
            e = cudaMemcpyAsync(phi, io->phi0_host, B * sizeof(double), cudaMemcpyHostToDevice, st);
        } else {
            fill_kernel<<<148, 256, 0, st>>>(phi, (long long)B, nan(""));
            e = cudaGetLastError();
        }
    }
    if (e != cudaSuccess) return cleanup(fail(IPMCMC_ECUDA, "host->device staging: %s", cudaGetErrorString(e)));
    ipmcmc_chain_buffers cb;
    memset(&cb, 0, sizeof cb);
    cb.u_dev = u;
    cb.phi_dev = phi;
    cb.model_state_dev = nvar ? mstate : nullptr;
    cb.mom_count_dev = cnt;
    cb.mom_mean_dev = mean;
    cb.mom_m2_dev = m2;
    cb.counters_dev = (int64_t *)counters;
    cb.trace_dev = io->samples_host ? trace : nullptr;
    cb.n_record = io->samples_host ? io->n_record : 0;
    if (n_sched) {   // the step queue's scratch in the arena, as ChainBatch passes its own
        cb.sched_dev = (int64_t *)sched;
        cb.sched_len = (int64_t)n_sched;
    }
    cb.sched_chunk = io->sched_chunk;
    rc = ipmcmc_run(p, s, &cb, n_chains, n_steps, stream);
    if (rc) return cleanup(rc);
    if (io->pooled_host) {
        rc = ipmcmc_pool_moments(n_chains, d, cnt, mean, m2, (const int64_t *)counters, pooled, pool_scratch, (int64_t)pool_bytes, stream);
        if (rc) return cleanup(rc);
    }
    if (io->samples_host) e = cudaMemcpyAsync(io->samples_host, trace, n_trace * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && io->u_host) e = cudaMemcpyAsync(io->u_host, u, B * d * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && io->phi_host) e = cudaMemcpyAsync(io->phi_host, phi, B * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && io->counters_host) e = cudaMemcpyAsync(io->counters_host, counters, B * CNT_N * sizeof(long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && io->pooled_host) e = cudaMemcpyAsync(io->pooled_host, pooled, (2 * d + 7) * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && nvar) e = cudaMemcpyAsync(io->model_state_host, mstate, B * nvar * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return cleanup(fail(IPMCMC_ECUDA, "run/device->host: %s", cudaGetErrorString(e)));
    return cleanup(0);
}

// ------------------------------------------------------------------------------------------------
// probes
// ------------------------------------------------------------------------------------------------
extern "C" int ipmcmc_lorenz_rhs(int32_t K, int32_t J, int32_t numerics, int64_t n, const double *theta_dev, const double *state_dev,
                                 double *rhs_dev, void *stream) {
    if (K < 1 || K > 32) return fail(IPMCMC_EUNSUPPORTED, "K=%d outside [1,32]", K);
    if (n <= 0) return 0;
    const int groups = lorenz_groups(K);
    const long long blocks = (n + groups - 1) / groups;
    LORENZ_DISPATCH(lorenz_rhs_kernel, J, K, numerics, <<<grid_for(blocks), 32, 0, (cudaStream_t)stream>>>(K, n, theta_dev, state_dev, rhs_dev));
    return 0;
}

extern "C" int ipmcmc_lorenz_rk45_attempt(int32_t K, int32_t J, int32_t numerics, int64_t n, const double *theta_dev,
                                          const double *state_dev, const double *h_dev, double rtol, double atol,
                                          double *out_dev, void *stream) {
    if (K < 1 || K > 32) return fail(IPMCMC_EUNSUPPORTED, "K=%d outside [1,32]", K);
    if (n <= 0) return 0;
    const int groups = lorenz_groups(K);
    const long long blocks = (n + groups - 1) / groups;
    LORENZ_DISPATCH(lorenz_attempt_kernel, J, K, numerics,
                    <<<grid_for(blocks), 32, 0, (cudaStream_t)stream>>>(K, n, theta_dev, state_dev, h_dev, rtol, atol, out_dev));
    return 0;
}

__global__ void rng_probe_kernel(unsigned long long seed, long long chain_offset, long long first_step,
                                 long long n_chains, long long n_steps, int d, double *out) {
    const long long total = n_chains * n_steps * (d + 1);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int slot = (int)(i % (d + 1));
        const long long s = (i / (d + 1)) % n_steps, c = i / ((long long)(d + 1) * n_steps);
        out[i] = slot < d ? draw_normal(seed, (uint64_t)(chain_offset + c), (uint64_t)(first_step + s), (uint32_t)slot)
                          : draw_uniform(seed, (uint64_t)(chain_offset + c), (uint64_t)(first_step + s));
    }
}

__global__ void div_probe_kernel(long long n, double a, const double *__restrict__ b, double *__restrict__ qf,
                                 double *__restrict__ qi) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        bool ok;
        qf[i] = BurgersWarp<1, NUM_EXACT, false>::div_rn_fast(a, b[i], ok);
        qi[i] = a / b[i];
    }
}
extern "C" int ipmcmc_div_probe(int64_t n, double a, const double *b_dev, double *q_fast_dev, double *q_ieee_dev, void *stream) {
    if (!b_dev || !q_fast_dev || !q_ieee_dev) return fail(IPMCMC_EINVAL, "NULL argument");
    if (n <= 0) return 0;
    div_probe_kernel<<<148 * 4, 256, 0, (cudaStream_t)stream>>>(n, a, b_dev, q_fast_dev, q_ieee_dev);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int ipmcmc_rng_probe(uint64_t seed, int64_t chain_offset, int64_t first_step, int64_t n_chains,
                                int64_t n_steps, int32_t dim, double *out_dev, void *stream) {
    if (!out_dev || dim < 1) return fail(IPMCMC_EINVAL, "bad argument");
    rng_probe_kernel<<<148 * 4, 256, 0, (cudaStream_t)stream>>>(seed, chain_offset, first_step, n_chains, n_steps, dim, out_dev);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// Dependent-free DFMA throughput: 8 independent FMA chains per thread, 2048 threads per SM.
__global__ void __launch_bounds__(256) dfma_peak_kernel(double *out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456) out[0] = s;
}

extern "C" int ipmcmc_fp64_peak(int32_t iters, double *tflops_out) {
    if (!tflops_out) return fail(IPMCMC_EINVAL, "NULL argument");
    int sms = 0;
    CUDA_TRY(sm_count(sms));
    double *out;
    CUDA_TRY(cudaMalloc((void **)&out, 8));
    const int inner = 2048, blocks = sms * 8;
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    dfma_peak_kernel<<<blocks, 256>>>(out, inner, 0.999999, 1e-9);  // warm-up
    double best = 0.0;
    for (int r = 0; r < (iters > 0 ? iters : 5); ++r) {
        CUDA_TRY(cudaEventRecord(e0));
        dfma_peak_kernel<<<blocks, 256>>>(out, inner, 0.999999, 1e-9);
        CUDA_TRY(cudaEventRecord(e1));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 8 * 16 * (double)inner * 256.0 * blocks;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    *tflops_out = best;
    return 0;
}
