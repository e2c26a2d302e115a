// Launchers of the Burgers kernels (definitions).  Included only by burgers_inst.cu, which is compiled
// once per cells-per-lane value (and once for the team kernels) so that the translation units build in
// parallel and ptxas sees each kernel family on its own; engine.cu sees the declarations only
// (burgers_launch.cuh).
#pragma once
#include <cstdlib>

#include "burgers_kernels.cuh"
#include "burgers_launch.cuh"

namespace ipmcmc {

#define IPMCMC_CU(expr)                               \
    do {                                              \
        const cudaError_t e_ = (expr);                \
        if (e_ != cudaSuccess) return e_;             \
    } while (0)

// kern<<<grid, block, smem, st>>>(args...), after raising the kernel's dynamic shared-memory limit when
// smem exceeds the 48 KB default.
template <class... P, class... A>
static cudaError_t launch(void (*kern)(P...), int grid, int block, size_t smem, cudaStream_t st, const A &...args) {
    if (smem > 48 * 1024) IPMCMC_CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, block, smem, st>>>(args...);
    return cudaGetLastError();
}

template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_forward(const BurgersDev &b, long long n, const double *u, double *G, double *phi,
                                  double *state, long long *work, cudaStream_t st) {
    // one chain per warp; CTAs of 4 warps (one per SM sub-partition) unless the batch is tiny
    int wpc = n >= 4 * 148 ? 4 : 1;
    if (const char *e = getenv("IPMCMC_FWD_WPC")) wpc = atoi(e) > 0 && atoi(e) <= 8 ? atoi(e) : wpc;  // experiments
    return launch(burgers_forward_kernel<CPL, NUM, PAD>, grid_for((n + wpc - 1) / wpc), 32 * wpc,
                  burgers_smem_bytes(b.N, wpc), st, b, n, u, G, phi, state, work);
}

template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_chain(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C, long long n_chains,
                                long long n_steps, int wpc, cudaStream_t st) {
    const long long slots = C.slot_chain ? (long long)C.n_slots : n_chains;
    return launch(burgers_chain_kernel<CPL, NUM, PAD>, grid_for((slots + wpc - 1) / wpc), 32 * wpc,
                  burgers_smem_bytes(b.N, wpc), st, b, S, C, n_chains, n_steps);
}

// Dynamic step scheduler (burgers_chain_queue_kernel): persistent warps, one wave.
template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_chain_queue(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C, long long n_chains,
                                      long long n_steps, int chunk, cudaStream_t st) {
    int n_sm = 148;
    IPMCMC_CU(sm_count(n_sm));
    // small batches: one CTA of W = ceil(n / n_SM) warps per SM (warp w -> sub-partition w % 4);
    // large batches: as many 4-warp CTAs as are resident at once (register and shared-memory limits).
    // Register budget (measured on B200, DESIGN.md section 6; tools/ab_bench.sh): up to 8 cells per lane the 128-register
    // build schedules the time step best at every batch size (1024 x 256: 67 % of the fp64 peak against
    // 61 % with 255 registers); from 16 cells per lane on it spills the state, and 255 registers with
    // half the resident warps win by far (8192 x 1024: 81 % against 66 %; 88 % with the rotated loop, which
    // only fits the 255-register build at 32 cells per lane).
    int wpc, grid;
    constexpr int MINB = CPL >= 16 ? 1 : 2;
    auto kern = burgers_chain_queue_kernel<CPL, NUM, PAD, MINB>;
    if (n_chains <= 8LL * n_sm) {
        wpc = (int)((n_chains + n_sm - 1) / n_sm);
        if (const char *e = getenv("IPMCMC_SCHED_WPC")) wpc = atoi(e) > 0 && atoi(e) <= 8 ? atoi(e) : wpc;  // experiments
        grid = (int)((n_chains + wpc - 1) / wpc);
        if (grid > n_sm) grid = n_sm;
        if (grid < n_sm && (long long)grid * wpc < n_chains) grid = n_sm;
    } else {
        // 4 warps of at most 1024 cells: within the default 48 KB of shared memory
        wpc = 4;
        int per_sm = 0;
        IPMCMC_CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * wpc, burgers_smem_bytes(b.N, wpc)));
        if (per_sm < 1) per_sm = 1;
        grid = per_sm * n_sm;
        const long long need = (n_chains + wpc - 1) / wpc;
        if (grid > need) grid = (int)need;
    }
    IPMCMC_CU(sched_init(C.sched, n_chains, st));
    return launch(kern, grid, 32 * wpc, burgers_smem_bytes(b.N, wpc), st, b, S, C, n_chains, n_steps, chunk);
}

// wide parameter vectors: CTAs of 4 warps (one per SM sub-partition) unless the batch is tiny, halved while
// their shared memory exceeds 200 KB
static int burgers_wide_warps(int N, int d, long long n) {
    int wpc = n >= 4 * 148 ? 4 : 1;
    while (wpc > 1 && burgers_wide_smem_bytes(N, d, wpc) > 200 * 1024) wpc /= 2;
    return wpc;
}
template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_wide_forward(const BurgersDev &b, long long n, const double *u, double *G, double *phi,
                                       double *state, long long *work, cudaStream_t st) {
    const int wpc = burgers_wide_warps(b.N, b.d, n);
    return launch(burgers_wide_forward_kernel<CPL, NUM, PAD>, grid_for((n + wpc - 1) / wpc), 32 * wpc,
                  burgers_wide_smem_bytes(b.N, b.d, wpc), st, b, n, u, G, phi, state, work);
}
template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_wide_chain(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C, long long n_chains,
                                     long long n_steps, cudaStream_t st) {
    const int wpc = burgers_wide_warps(b.N, S.d, n_chains);
    return launch(burgers_wide_chain_kernel<CPL, NUM, PAD>, grid_for((n_chains + wpc - 1) / wpc), 32 * wpc,
                  burgers_wide_smem_bytes(b.N, S.d, wpc), st, b, S, C, n_chains, n_steps);
}

template <int NUM, int TM>
cudaError_t burgers_launch_team_forward(const BurgersDev &b, long long n, const double *u, double *G, double *phi,
                                       double *state, long long *work, cudaStream_t st) {
    return launch(burgers_team_forward_kernel<32, NUM, TM>, grid_for(n), 32 * TM, burgers_team_smem_bytes(b.N), st,
                  b, n, u, G, phi, state, work);
}
template <int NUM, int TM>
cudaError_t burgers_launch_team_chain(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C, long long n_chains,
                                     long long n_steps, cudaStream_t st) {
    return launch(burgers_team_chain_kernel<32, NUM, TM>, grid_for(n_chains), 32 * TM, burgers_team_smem_bytes(b.N), st,
                  b, S, C, n_chains, n_steps);
}

}  // namespace ipmcmc
