// Launchers of the Burgers kernels (declarations; definitions in burgers_launch_impl.cuh, explicit
// instantiations in burgers_inst.cu).  They return the CUDA status of the launch.
#pragma once
#include <cuda_runtime.h>

#include "burgers.cuh"
#include "sampler.cuh"

namespace ipmcmc {

template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_forward(const BurgersDev &b, long long n, const double *u, double *G, double *phi,
                                   double *state, long long *work, cudaStream_t st);
template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_chain_queue(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C,
                                       long long n_chains, long long n_steps, int chunk, cudaStream_t st);
template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_wide_forward(const BurgersDev &b, long long n, const double *u, double *G, double *phi,
                                        double *state, long long *work, cudaStream_t st);
template <int CPL, int NUM, bool PAD>
cudaError_t burgers_launch_wide_chain(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C, long long n_chains,
                                      long long n_steps, cudaStream_t st);
template <int NUM, int TM>
cudaError_t burgers_launch_team_forward(const BurgersDev &b, long long n, const double *u, double *G, double *phi,
                                        double *state, long long *work, cudaStream_t st);
template <int NUM, int TM>
cudaError_t burgers_launch_team_chain(const BurgersDev &b, const SamplerDev &S, const ChainBufDev &C,
                                      long long n_chains, long long n_steps, cudaStream_t st);

}  // namespace ipmcmc
