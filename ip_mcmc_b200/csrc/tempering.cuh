// Replica exchange (parallel tempering) between the rungs of ladders of Burgers chains.
// A tempered batch is n_ladders x K chains, ladder-major: local chain l*K + k is rung k of ladder l, whose
// likelihood the Metropolis step tempers by inv_temp[l*K + k] (metropolis_step, burgers_kernels.cuh).
// Round r proposes the pairs (k, k+1) with k = r (mod 2) in every ladder (deterministic even-odd pairing,
// Syed et al., JRSS-B 2022) and swaps the two states iff
//     exp((t_k - t_{k+1}) * (Phi_k - Phi_{k+1})) > U,
// U = Philox (seed, global id of slot k) at (step r, slot SLOT_SWAP).  The prior and the RW regulariser are
// common to all rungs and cancel.  u rows, Phi and the replica records move; moments, counters and traces
// stay with the slot.
// CPU statement: oracle/tempering_np.py.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace ipmcmc {

// No chain draw uses this slot: proposal normals use slots < d <= 256, the accept uniform SLOT_UNIFORM.
constexpr uint32_t SLOT_SWAP = 0xFFFFFFFEu;

struct SwapDev {
    long long n_ladders, chain_offset, round;
    int K, d, n_pairs, parity;   // n_pairs proposed per ladder this round, k = parity + 2 * pair
    unsigned long long seed;
    double *u, *phi;
    const double *inv_temp, *inject_u;   // inject_u: [n_ladders, K-1] uniform of pair (k, k+1), or nullptr
    int *replica;                        // [B, 2] (replica id, direction)
    long long *swap_counts;              // [n_ladders, K-1, 2] (attempts, accepts)
    long long *round_trips;              // [n_ladders]
};

// One warp per proposed pair: lane 0 decides and keeps the books, the lanes exchange the u rows.
__global__ void __launch_bounds__(256) swap_round_kernel(const __grid_constant__ SwapDev W) {
    const long long n = W.n_ladders * W.n_pairs;
    const int lane = lane_id();
    for (long long p = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < n;
         p += ((long long)gridDim.x * blockDim.x) >> 5) {
        const long long l = p / W.n_pairs;
        const int k = W.parity + 2 * (int)(p % W.n_pairs);
        const long long a = l * W.K + k, b = a + 1;   // local chain ids of rungs k and k+1
        int swap = 0;
        if (lane == 0) {
            const double acc = exp((W.inv_temp[a] - W.inv_temp[b]) * (W.phi[a] - W.phi[b]));
            const double U = W.inject_u ? W.inject_u[l * (W.K - 1) + k]
                                        : draw_uniform(W.seed, (uint64_t)(W.chain_offset + a), (uint64_t)W.round, SLOT_SWAP);
            swap = acc > U;   // strict; NaN compares false
            long long *sc = W.swap_counts + (l * (W.K - 1) + k) * 2;
            sc[0] += 1;
            sc[1] += swap;
        }
        swap = __shfl_sync(FULL, swap, 0);
        if (swap) {
            for (int i = lane; i < W.d; i += 32) {
                const double x = W.u[a * W.d + i];
                W.u[a * W.d + i] = W.u[b * W.d + i];
                W.u[b * W.d + i] = x;
            }
        }
        if (lane == 0) {
            if (swap) {
                const double ph = W.phi[a];
                W.phi[a] = W.phi[b];
                W.phi[b] = ph;
                for (int j = 0; j < 2; ++j) {
                    const int r = W.replica[2 * a + j];
                    W.replica[2 * a + j] = W.replica[2 * b + j];
                    W.replica[2 * b + j] = r;
                }
            }
            // a replica that went up to the hottest rung and is back at t = 1 has made a round trip
            if (k == 0) {
                int *r0 = W.replica + 2 * (l * W.K);
                if (r0[1] == -1) W.round_trips[l] += 1;
                r0[1] = 1;
            }
            if (k + 1 == W.K - 1) W.replica[2 * (l * W.K + W.K - 1) + 1] = -1;
        }
    }
}

}  // namespace ipmcmc
