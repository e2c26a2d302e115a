// Shared device helpers.  The whole library is compiled with -fmad=false: every FMA in the
// generated code is an explicit fma() (the FUSED numerics and the CUDA math library), so the
// EXACT paths reproduce the reference's floating-point operation order bit for bit.
#pragma once
#include <stdint.h>
#include <cuda_runtime.h>

#include "../../include/ipmcmc.h"

namespace ipmcmc {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// Developer instrumentation (-DIPMCMC_PROF=1, tools/overhead_probe.py): cycles per section of a work
// item, summed over all warps by lane 0.  Not compiled into the product library.
#ifndef IPMCMC_PROF
#define IPMCMC_PROF 0
#endif
#if IPMCMC_PROF
static __device__ unsigned long long g_prof[16];
#define PROF_T(var) const long long var = clock64()
#define PROF_ADD(slot, a, b) do { if (lane_id() == 0) atomicAdd(&g_prof[slot], (unsigned long long)((b) - (a))); } while (0)
#else
#define PROF_T(var)
#define PROF_ADD(slot, a, b)
#endif

// grid.x for n_blocks CTAs (clamped to the largest grid.x; the kernels stride over the rest)
inline int grid_for(long long n_blocks) { return (int)(n_blocks < 2147483647LL ? n_blocks : 2147483647LL); }

// number of SMs of the current device
inline cudaError_t sm_count(int &n_sm) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    return e;
}

// 64-bit shuffles
__device__ __forceinline__ double shfl(double v, int src, unsigned mask = FULL) { return __shfl_sync(mask, v, src); }
__device__ __forceinline__ double shfl_up1(double v) { return __shfl_up_sync(FULL, v, 1); }
__device__ __forceinline__ double shfl_down1(double v) { return __shfl_down_sync(FULL, v, 1); }

// sum over the warp in a fixed order (lane tree), the same bits on every lane
__device__ __forceinline__ double warp_sum_fixed(double v) {
#pragma unroll
    for (int off = 1; off < 32; off *= 2) {
        const double o = __shfl_xor_sync(FULL, v, off);
        v = (lane_id() & off) ? o + v : v + o;
    }
    return v;
}

// (count, mean, M2) and Chan et al.'s merge of two such triples
struct Mom3 {
    double n, mean, m2;
};
__device__ __forceinline__ Mom3 chan_merge(const Mom3 &a, const Mom3 &b) {
    const double nt = a.n + b.n;
    if (!(nt > 0.0)) return Mom3{0.0, 0.0, 0.0};
    const double delta = b.mean - a.mean;
    return Mom3{nt, a.mean + delta * (b.n / nt), (a.m2 + b.m2) + delta * delta * (a.n * b.n / nt)};
}

// |x| as an ordered 64-bit integer key: IEEE-754 ordering of non-negative doubles equals the
// ordering of their bit patterns.  Kept in integer registers on purpose -- a round trip through
// double makes the compiler re-materialise fabs as a DADD on the (precious) fp64 pipe.
__device__ __forceinline__ uint64_t abs_key(double v) {
    return ((uint64_t)((uint32_t)__double2hiint(v) & 0x7fffffffu) << 32) | (uint32_t)__double2loint(v);
}
__device__ __forceinline__ uint64_t key_max(uint64_t a, uint64_t b) { return a > b ? a : b; }

// max over the warp of 64-bit keys on the integer REDUX unit (2 x CREDUX.MAX) instead of 5
// shuffle + DSETP rounds on the fp64 pipe.
__device__ __forceinline__ double warp_max_key(uint64_t k) {
    const uint32_t hi = (uint32_t)(k >> 32), lo = (uint32_t)k;
    const uint32_t mh = __reduce_max_sync(FULL, hi);
    const uint32_t ml = __reduce_max_sync(FULL, hi == mh ? lo : 0u);
    return __hiloint2double((int)mh, (int)ml);
}

// max(|a|,|b|) for doubles through the integer pipe (keeps the fp64 pipe for arithmetic).
__device__ __forceinline__ double absmax_bits(double a, double b) {
    const uint64_t m = key_max(abs_key(a), abs_key(b));
    return __hiloint2double((int)(m >> 32), (int)(uint32_t)m);
}

// NumPy's pairwise summation (numpy/_core/src/umath/loops_utils.h.src, @TYPE@_pairwise_sum) of
// f(start), ..., f(start+n-1); restated in oracle/burgers_np.py:np_pairwise_sum.  The reference's
// np.trapz (utilities.py:107), np.sum in scipy's logpdf and np.mean reduce in exactly this order.
template <class F>
__device__ double np_pairwise_sum(const F &f, int start, int n) {
    if (n < 8) {
        double res = -0.0;
        for (int i = 0; i < n; ++i) res = res + f(start + i);
        return res;
    }
    if (n <= 128) {
        double r[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = f(start + k);
        int i = 8;
        for (; i < n - (n % 8); i += 8) {
#pragma unroll
            for (int k = 0; k < 8; ++k) r[k] = r[k] + f(start + i + k);
        }
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; ++i) res = res + f(start + i);
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    return np_pairwise_sum(f, start, n2) + np_pairwise_sum(f, start + n2, n - n2);
}

// Gaussian-misfit potential constants (device copy of ipmcmc_potential_desc)
struct PotentialDev {
    int q;
    int dense;
    double log_const;
    double y[IPMCMC_MAX_OBS];
    double scale[IPMCMC_MAX_OBS];
    int perm[IPMCMC_MAX_OBS];
    const double *LP;  // device, dense only
};

// Phi = 0.5*((rank*log2pi + logdet) + sum_i r_i^2), r = (y - G) @ LP   (potential.py:53-54 via
// scipy _multivariate.py:585-591).  G lives in shared memory scratch g[q]; every lane computes
// the same value (broadcast reads), so no shuffle is needed afterwards.  `r2` is scratch [q].
__device__ __forceinline__ double potential_from_G(const PotentialDev &P, const double *g, double *r2,
                                                   int lane, int group_lanes, unsigned mask) {
    for (int i = lane; i < P.q; i += group_lanes) {
        double r;
        if (!P.dense) {
            const int j = P.perm[i];
            r = (P.y[j] - g[j]) * P.scale[i];
        } else {
            r = 0.0;
            for (int j = 0; j < P.q; ++j) r = r + (P.y[j] - g[j]) * P.LP[j * P.q + i];
        }
        r2[i] = r * r;
    }
    __syncwarp(mask);
    const double maha = np_pairwise_sum([&](int i) { return r2[i]; }, 0, P.q);
    __syncwarp(mask);
    return 0.5 * (P.log_const + maha);
}

}  // namespace ipmcmc
