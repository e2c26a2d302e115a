// Convergence diagnostics over a recorded trace (DESIGN.md section 4.3): element (c, i, j) of chain c, draw i,
// parameter j is x[c * cs + i * d + j] for a chain stride cs >= n * d, so that a view trace[:, burn:] is read
// in place.  The estimators are restated on the host in ip_mcmc_b200/stats.py (integrated_autocorr_time,
// split_rhat, multichain_ess), which the tests compare against.
//
// Every sum below has an order fixed by (M, n, d) alone: per-series sums are lane-strided partial sums
// reduced by warp_sum_fixed, and sums over chains are trees over fixed chain chunks merged in chunk order
// (as pool_partial_kernel / pool_final_kernel).  Staging in shared memory or reading through L2 gives
// the same bits, so results do not depend on the launch geometry or the device.
#pragma once
#include "common.cuh"

namespace ipmcmc {

constexpr int DIAG_SMEM = 200 * 1024;   // dynamic shared memory a diagnostics CTA may stage series in
constexpr int DIAG_WARPS = 8;           // warps per CTA of the sequence and variogram kernels
constexpr int SEQ_CHUNK = 64;           // chains per CTA of the sequence statistics
constexpr int VARIO_BLOCKS = 128;       // chain chunks of the variogram sums (at most)

// chains per chunk of the variogram sums: at most VARIO_BLOCKS chunks of at least 8 chains
__host__ __device__ inline long long vario_chunk(long long M) {
    const long long c = (M + VARIO_BLOCKS - 1) / VARIO_BLOCKS;
    return c < 8 ? 8 : c;
}

// ---- A. per-chain integrated autocorrelation time (stats.integrated_autocorr_time) ---------------------
// One warp per series (c, j).  y = x - mean is staged in the warp's shared memory when it fits (STAGED) and
// recomputed from the trace otherwise.  Geyer's initial positive sequence: each pass of the lag loop
// computes rho_k and rho_{k+1} and the warp stops at its own series' cut-off, O(n * tau) per series.
template <bool STAGED>
__global__ void __launch_bounds__(256) diag_tau_kernel(long long M, long long n, int d, const double *__restrict__ x,
                                                       long long cs, double *__restrict__ tau) {
    extern __shared__ double sm[];
    const int lane = lane_id(), w = threadIdx.x >> 5, W = blockDim.x >> 5;
    double *ys = sm + (long long)w * n;
    for (long long sr = (long long)blockIdx.x * W + w; sr < M * d; sr += (long long)gridDim.x * W) {
        const long long c = sr / d;
        const int j = (int)(sr - c * d);
        const double *xs = x + c * cs + j;   // draw i at xs[i * d]
        const double x0 = xs[0];
        double s = 0.0;
        bool same = true;
        for (long long i = lane; i < n; i += 32) {
            const double v = xs[i * d];
            s += v;
            same = same && v == x0;
        }
        // A series stuck at one value (a chain that accepted nothing) takes its mean in NumPy's pairwise order, as
        // stats.autocorr does: whether y = x - mean is exactly zero (the all-ones case below) or a constant rounding
        // residue depends on that order, and tau differs by a factor of about 2 between the two.
        const double mean = __all_sync(FULL, same) ? np_pairwise_sum([&](int) { return x0; }, 0, (int)n) / (double)n
                                                   : warp_sum_fixed(s) / (double)n;
        double g = 0.0;
        for (long long i = lane; i < n; i += 32) {
            const double y = xs[i * d] - mean;
            if (STAGED) ys[i] = y;
            g = fma(y, y, g);
        }
        const double g0 = warp_sum_fixed(g);
        __syncwarp();
        auto Y = [&](long long i) { return STAGED ? ys[i] : xs[i * d] - mean; };
        double t;
        if (g0 == 0.0) {
            t = 1.0 + 4.0 * (double)((n - 1) / 2);   // stats.autocorr: all ones for a constant series
        } else {
            t = 1.0;
            for (long long k = 1; k + 1 < n; k += 2) {
                double a = 0.0, b = 0.0;
                for (long long i = lane; i + k < n; i += 32) {
                    const double yi = Y(i);
                    a = fma(yi, Y(i + k), a);
                    if (i + k + 1 < n) b = fma(yi, Y(i + k + 1), b);
                }
                const double pair = warp_sum_fixed(a) / g0 + warp_sum_fixed(b) / g0;
                if (pair <= 0.0) break;   // a NaN pair does not stop the sum, as on the host
                t += 2.0 * pair;
            }
            t = t < 1.0 ? 1.0 : t;
        }
        if (lane == 0) tau[c * d + j] = t;
        __syncwarp();
    }
}

// ---- B. split-sequence statistics -------------------------------------------------------------------
// Sequence 2c is draws [0, h) of chain c, sequence 2c+1 draws [n-h, n) (h = n/2; the middle draw of an odd
// n is dropped).  Pass 1: CTA (b, j) takes chains [b*SEQ_CHUNK, (b+1)*SEQ_CHUNK); warp w takes sequences
// w, w+8, ... of the chunk, computes each one's mean and ddof=1 variance (two passes, warp_sum_fixed), and
// merges (1, mean, 0) into its (n, mean, M2) with Chan's formula and adds the variance; the 8 warps are
// merged in order -> partial[b][j] = (m, mean of the sequence means, M2 of the sequence means, sum s^2).
// Pass 2 merges the chunks in order.
__global__ void __launch_bounds__(DIAG_WARPS * 32) diag_seq_partial_kernel(long long M, long long n, int d,
                                                                          const double *__restrict__ x, long long cs,
                                                                          double *__restrict__ partial) {   // [nb, d, 4]
    __shared__ double red[DIAG_WARPS][4];
    const int lane = lane_id(), w = threadIdx.x >> 5, j = blockIdx.y;
    const long long h = n / 2;
    const long long c0 = (long long)blockIdx.x * SEQ_CHUNK;
    const long long c1 = c0 + SEQ_CHUNK < M ? c0 + SEQ_CHUNK : M;
    Mom3 acc{0.0, 0.0, 0.0};
    double s2 = 0.0;
    for (long long s = 2 * c0 + w; s < 2 * c1; s += DIAG_WARPS) {
        const double *xs = x + (s >> 1) * cs + ((s & 1) ? n - h : 0) * d + j;
        double a = 0.0;
        for (long long i = lane; i < h; i += 32) a += xs[i * d];
        const double mean = warp_sum_fixed(a) / (double)h;
        double q = 0.0;
        for (long long i = lane; i < h; i += 32) {
            const double y = xs[i * d] - mean;
            q = fma(y, y, q);
        }
        const double var = warp_sum_fixed(q) / (double)(h - 1);
        acc = chan_merge(acc, Mom3{1.0, mean, 0.0});
        s2 += var;
    }
    if (lane == 0) {
        red[w][0] = acc.n;
        red[w][1] = acc.mean;
        red[w][2] = acc.m2;
        red[w][3] = s2;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        Mom3 r{0.0, 0.0, 0.0};
        double t = 0.0;
        for (int k = 0; k < DIAG_WARPS; ++k) {
            r = chan_merge(r, Mom3{red[k][0], red[k][1], red[k][2]});
            t += red[k][3];
        }
        double *o = partial + ((long long)blockIdx.x * d + j) * 4;
        o[0] = r.n;
        o[1] = r.mean;
        o[2] = r.m2;
        o[3] = t;
    }
}

__global__ void __launch_bounds__(64) diag_seq_final_kernel(int nb, int d, const double *__restrict__ partial,
                                                           double *__restrict__ out) {   // [d, 4]
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        Mom3 r{0.0, 0.0, 0.0};
        double t = 0.0;
        for (int b = 0; b < nb; ++b) {
            const double *p = partial + ((long long)b * d + j) * 4;
            r = chan_merge(r, Mom3{p[0], p[1], p[2]});
            t += p[3];
        }
        out[4 * j + 0] = r.n;
        out[4 * j + 1] = r.mean;
        out[4 * j + 2] = r.m2;
        out[4 * j + 3] = t;
    }
}

// ---- C. variogram sums  V[j][t] = sum_s sum_{i=t}^{h-1} (psi_{s,i} - psi_{s,i-t})^2, t in [t0, t0 + L) -----
// Pass 1: CTA (b, g, j) takes the chains of chunk b (vario_chunk(M) chains) and lags t0 + 32g + lane; warp w
// takes sequences w, w+8, ... of the chunk, stages each one in its shared memory (STAGED) or reads it through
// L2, and lane l adds (psi_{q+t} - psi_q)^2 over q = 0 .. h-1-t (psi_q is a broadcast read, psi_{q+t} a
// consecutive one) in two interleaved accumulators.  The 8 warps are added in order.  Parameters whose
// truncation is already decided (done[j] != 0) are skipped.  Pass 2 adds the chunks in order.
template <bool STAGED>
__global__ void __launch_bounds__(DIAG_WARPS * 32) diag_vario_partial_kernel(long long M, long long n, int d,
                                                                            const double *__restrict__ x, long long cs,
                                                                            long long t0, long long L,
                                                                            const int *__restrict__ done,
                                                                            double *__restrict__ partial) {   // [nb, d, L]
    extern __shared__ double sm[];
    __shared__ double red[DIAG_WARPS][32];
    const int lane = lane_id(), w = threadIdx.x >> 5, j = blockIdx.z;
    if (done && done[j]) return;
    const long long h = n / 2, chunk = vario_chunk(M);
    const long long c0 = (long long)blockIdx.x * chunk;
    const long long c1 = c0 + chunk < M ? c0 + chunk : M;
    const long long t = t0 + 32LL * blockIdx.y + lane;
    double *ps = sm + (long long)w * h;
    double acc = 0.0;
    for (long long s = 2 * c0 + w; s < 2 * c1; s += DIAG_WARPS) {
        const double *xs = x + (s >> 1) * cs + ((s & 1) ? n - h : 0) * d + j;
        if (STAGED) {
            for (long long i = lane; i < h; i += 32) ps[i] = xs[i * d];
            __syncwarp();
        }
        auto P = [&](long long i) { return STAGED ? ps[i] : xs[i * d]; };
        const long long cnt = h - t;   // <= 0 for lags past the end
        double a0 = 0.0, a1 = 0.0;
        long long q = 0;
        for (; q + 1 < cnt; q += 2) {
            const double e0 = P(q + t) - P(q), e1 = P(q + 1 + t) - P(q + 1);
            a0 = fma(e0, e0, a0);
            a1 = fma(e1, e1, a1);
        }
        if (q < cnt) {
            const double e0 = P(q + t) - P(q);
            a0 = fma(e0, e0, a0);
        }
        acc += a0 + a1;
        __syncwarp();
    }
    red[w][lane] = acc;
    __syncthreads();
    if (threadIdx.x < 32 && t < t0 + L) {
        double r = 0.0;
        for (int k = 0; k < DIAG_WARPS; ++k) r += red[k][threadIdx.x];
        partial[((long long)blockIdx.x * d + j) * L + (t - t0)] = r;
    }
}

__global__ void __launch_bounds__(128) diag_vario_final_kernel(int nb, int d, long long L, const double *__restrict__ partial,
                                                              const int *__restrict__ done, double *__restrict__ out,
                                                              long long ld) {   // out[j * ld + (t - t0)]
    const int j = blockIdx.y;
    if (done && done[j]) return;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < L; k += (long long)gridDim.x * blockDim.x) {
        double r = 0.0;
        for (int b = 0; b < nb; ++b) r += partial[((long long)b * d + j) * L + k];
        out[(long long)j * ld + k] = r;
    }
}

// ---- truncation and final R-hat / n_eff / T (stats.split_rhat, stats.multichain_ess) ----------------
// One thread per parameter advances the truncated sum over the lags [1, lag_end) summed so far.  state[j] =
// (S, t) holds the loop between calls (zero before the first); the loop pauses before `S += rho_t` when a
// lag it needs (up to t+2, which may fall into the next block) is not summed yet, so the sums and the
// decision are the host loop's whatever the block boundaries.  When the loop ends, out = (R-hat [d],
// n_eff [d], T [d]) and done[j] = 1.
__global__ void __launch_bounds__(64) diag_truncate_kernel(long long h, int d, const double *__restrict__ seq,
                                                          const double *__restrict__ vsum, long long ld, long long lag_end,
                                                          double *__restrict__ state, int *__restrict__ done,
                                                          double *__restrict__ out) {
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        if (done[j]) continue;
        const double m = seq[4 * j], m2 = seq[4 * j + 2], s2 = seq[4 * j + 3], hd = (double)h;
        const double W = s2 / m, B = hd / (m - 1.0) * m2;
        const double varp = (hd - 1.0) / hd * W + B / hd;
        const double *v = vsum + (long long)j * ld;
        auto rho = [&](long long t) { return 1.0 - v[t] / (m * (double)(h - t)) / (2.0 * varp); };
        double S = state[2 * j];
        long long t = state[2 * j + 1] == 0.0 ? 1 : (long long)state[2 * j + 1];
        bool fin = false;
        for (;;) {
            const bool last = t + 2 > h - 1;
            if ((last ? t : t + 2) >= lag_end) break;
            S += rho(t);
            if (last || rho(t + 1) + rho(t + 2) < 0.0) {
                fin = true;
                break;
            }
            S += rho(t + 1);
            t += 2;
        }
        state[2 * j] = S;
        state[2 * j + 1] = (double)t;
        if (fin) {
            out[j] = sqrt(varp / W);
            out[d + j] = m * hd / (1.0 + 2.0 * S);
            out[2 * d + j] = (double)t;
            done[j] = 1;
        }
    }
}

}  // namespace ipmcmc
