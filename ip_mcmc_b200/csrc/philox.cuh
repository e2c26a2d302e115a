// Counter-based RNG of the engine: Philox4x32-10 keyed by (seed, global chain id), counted by
// (step, slot).  Replaces the reference's single shared numpy Generator (burgers_mcmc.py:101,
// lorenz_mcmc.py:83; "only one source of randomness", report/code.org:12) whose draw ORDER is
// part of its behaviour; counter-based draws are order-free and invariant to the GPU count.
// CPU statement: oracle/philox_np.py (bit-exact for the integers, <= few ulp for the normals).
#pragma once
#include <stdint.h>

namespace ipmcmc {

constexpr uint32_t PHILOX_M0 = 0xD2511F53u;
constexpr uint32_t PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u;
constexpr uint32_t PHILOX_W1 = 0xBB67AE85u;
constexpr uint32_t SLOT_UNIFORM = 0xFFFFFFFFu;

struct Philox4 {
    uint32_t x0, x1, x2, x3;
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                 uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(PHILOX_M0, c0), lo0 = PHILOX_M0 * c0;
        const uint32_t hi1 = __umulhi(PHILOX_M1, c2), lo1 = PHILOX_M1 * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += PHILOX_W0;
        k1 += PHILOX_W1;
    }
    return Philox4{c0, c1, c2, c3};
}

__device__ __forceinline__ Philox4 draw_words(uint64_t seed, uint64_t chain, uint64_t step, uint32_t slot) {
    return philox4x32_10((uint32_t)step, (uint32_t)(step >> 32), slot, (uint32_t)(seed >> 32),
                         (uint32_t)seed, (uint32_t)chain);
}

// U in [0,1): the 53-bit mapping numpy's Generator.random() uses ((x >> 11) * 2^-53).  The accept uniform
// uses SLOT_UNIFORM, the replica-exchange uniform SLOT_SWAP (tempering.cuh).
__device__ __forceinline__ double draw_uniform(uint64_t seed, uint64_t chain, uint64_t step,
                                               uint32_t slot = SLOT_UNIFORM) {
    const Philox4 r = draw_words(seed, chain, step, slot);
    const uint64_t x = ((uint64_t)r.x1 << 32) | r.x0;
    return (double)(x >> 11) * 0x1.0p-53;
}

// Standard normal by Box-Muller: sqrt(-2 ln u1) cos(2 pi u2), u1 in (0,1], u2 in [0,1).
__device__ __forceinline__ double draw_normal(uint64_t seed, uint64_t chain, uint64_t step, uint32_t slot) {
    const Philox4 r = draw_words(seed, chain, step, slot);
    const uint64_t a = ((uint64_t)r.x1 << 32) | r.x0;
    const uint64_t b = ((uint64_t)r.x3 << 32) | r.x2;
    const double u1 = (double)((a >> 11) + 1ull) * 0x1.0p-53;
    const double u2 = (double)(b >> 11) * 0x1.0p-53;
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
}

}  // namespace ipmcmc
