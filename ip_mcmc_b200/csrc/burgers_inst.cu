// Explicit instantiations of the Burgers launchers (and with them the kernels) for ONE cells-per-lane
// value and ONE numerics: compiled as  nvcc -DIPMCMC_TU_CPL=<1|2|4|7|8|16|32> -DIPMCMC_TU_NUM=<0 exact|1 fused>
// -c burgers_inst.cu  (CPL 0 = the team kernels for 2048 / 4096 cells, both numerics), see ip_mcmc_b200/build.py.
#include "burgers_launch_impl.cuh"

#ifndef IPMCMC_TU_CPL
#error "compile with -DIPMCMC_TU_CPL=<cells per lane> (0 = team kernels)"
#endif

namespace ipmcmc {

#if IPMCMC_TU_CPL > 0
#define INST(NUM, PAD)                                                                                              \
    template cudaError_t burgers_launch_forward<IPMCMC_TU_CPL, NUM, PAD>(const BurgersDev &, long long, const double *, \
                                                                         double *, double *, double *, long long *,  \
                                                                         cudaStream_t);                              \
    template cudaError_t burgers_launch_chain_queue<IPMCMC_TU_CPL, NUM, PAD>(const BurgersDev &, const SamplerDev &,    \
                                                                             const ChainBufDev &, long long, long long, \
                                                                             int, cudaStream_t);                     \
    template cudaError_t burgers_launch_wide_forward<IPMCMC_TU_CPL, NUM, PAD>(const BurgersDev &, long long,            \
                                                                              const double *, double *, double *,     \
                                                                              double *, long long *, cudaStream_t);   \
    template cudaError_t burgers_launch_wide_chain<IPMCMC_TU_CPL, NUM, PAD>(const BurgersDev &, const SamplerDev &,     \
                                                                            const ChainBufDev &, long long, long long, \
                                                                            cudaStream_t);
#if !defined(IPMCMC_TU_NUM) || IPMCMC_TU_NUM == 0
INST(NUM_EXACT, false)
INST(NUM_EXACT, true)
#endif
#if !defined(IPMCMC_TU_NUM) || IPMCMC_TU_NUM == 1
INST(NUM_FUSED, false)
INST(NUM_FUSED, true)
#endif
#else
#define INST(NUM, TM)                                                                                             \
    template cudaError_t burgers_launch_team_forward<NUM, TM>(const BurgersDev &, long long, const double *, double *, \
                                                              double *, double *, long long *, cudaStream_t);        \
    template cudaError_t burgers_launch_team_chain<NUM, TM>(const BurgersDev &, const SamplerDev &, const ChainBufDev &, \
                                                            long long, long long, cudaStream_t);
INST(NUM_EXACT, 2)
INST(NUM_EXACT, 4)
INST(NUM_FUSED, 2)
INST(NUM_FUSED, 4)
#endif

}  // namespace ipmcmc

#if IPMCMC_PROF && IPMCMC_TU_CPL == 8
// developer instrumentation only (tools/overhead_probe.py); not declared in include/ipmcmc.h
extern "C" int ipmcmc_prof_read(unsigned long long *out16, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out16, ipmcmc::g_prof, sizeof(unsigned long long) * 16);
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(ipmcmc::g_prof, z, sizeof(z));
    }
    return 0;
}
#endif
