// Dynamic step scheduler shared by the Burgers and the Lorenz chain kernels: a FIFO of READY work
// units (a chain, or a warp's group of Lorenz chains) in global memory, served by persistent warps.
#pragma once
#include "common.cuh"

namespace ipmcmc {

// ------------------------------------------------------------------------------------------------
// Dynamic step scheduler.  Solve lengths are data dependent and the warps of an SM do not all run
// at the same speed (a warp alone on a sub-partition advances ~1.85x faster than one that shares
// it), so a static chain -> warp map leaves sub-partitions idle at the end of a launch.  Here
// persistent warps take (chain, `chunk` steps) work items from a FIFO of READY chains in global
// memory: a chain is pushed back as soon as its item is done, so chains rotate over the warps,
// advance at the same average pace and every warp stays busy until the queue runs dry.  The chain
// state (u, Phi, moments: ~100 B) travels through L2 between items; Philox is keyed by (chain,
// step), so the results do not depend on which warp ran which item: the same bits for any chunk,
// CTA shape and launch split (tests/test_gpu_chains.py, test_queue_is_pure_scheduling;
// tests/test_gpu_lorenz.py, test_lorenz_queue_is_pure_scheduling).
//
// Scratch (int64, the caller's or a stream-ordered allocation of the library): ring[cap] | progress[n] | head | tail, cap = 2*n (n = work units).
// Ring entry = ((lap+1) << 32) | chain for the ticket lap*cap + slot; 0 = consumed/empty.
// ------------------------------------------------------------------------------------------------
struct SchedView {
    unsigned long long *ring, *head, *tail;
    long long *progress;
    long long cap;
    __device__ __forceinline__ SchedView(long long *base, long long n_chains)
        : ring((unsigned long long *)base), head((unsigned long long *)base + 3 * n_chains),
          tail((unsigned long long *)base + 3 * n_chains + 1), progress(base + 2 * n_chains), cap(2 * n_chains) {}
};
__host__ __device__ inline long long sched_len(long long n_chains) { return 3 * n_chains + 2; }

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

static __global__ void sched_init_kernel(long long *sched, long long n_chains) {
    SchedView Q(sched, n_chains);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < Q.cap; i += (long long)gridDim.x * blockDim.x) {
        Q.ring[i] = i < n_chains ? ((1ull << 32) | (unsigned long long)i) : 0ull;
        if (i < n_chains) Q.progress[i] = 0;
        if (i == 0) {
            *Q.head = 0;
            *Q.tail = (unsigned long long)n_chains;
        }
    }
}

// Queues work units 0 .. n_units - 1, each at step 0, on stream st (ahead of the kernel that serves them).
static inline cudaError_t sched_init(long long *sched, long long n_units, cudaStream_t st) {
    const long long blocks = (2 * n_units + 255) / 256;
    sched_init_kernel<<<(unsigned)(blocks < 1184 ? blocks : 1184), 256, 0, st>>>(sched, n_units);
    return cudaGetLastError();
}

// Spin until lane 0 reads a value accepted by `ok` from *p; returns it on every lane.  The loop
// condition is warp-uniform (lane 0 only issues a predicated load): a lane spinning on its own
// does not reconverge with the other 31, and the whole solve would then run twice, once per part
// of the split warp (measured: 4x slower).
template <class OK>
__device__ __forceinline__ unsigned long long spin_until(const unsigned long long *p, int lane, OK ok) {
    while (true) {
        unsigned long long v = 0;
        if (lane == 0) v = ld_acquire_u64(p);
        v = __shfl_sync(FULL, v, 0);
        if (ok(v)) return v;
        __nanosleep(64);
    }
}

// Global loads/stores of the chain state.  Under the dynamic scheduler (QUEUE) another SM may have
// written the state earlier in the same launch: go through L2 (L1 is not coherent).
template <bool QUEUE, class T>
__device__ __forceinline__ T ld_state(const T *p) { return QUEUE ? __ldcg(p) : *p; }
template <bool QUEUE, class T>
__device__ __forceinline__ void st_state(T *p, T v) {
    if (QUEUE) __stcg(p, v);
    else *p = v;
}

// The warp's serving loop, called by all 32 lanes: take a ticket, wait for its ring slot, consume it,
// run `body(unit, s0, s1)` (steps [s0, s1) of the launch for that work unit, `chunk` at most), and push
// the unit back while it has steps left; returns when every item has been taken.
// The unit's state -- what `body` stored with st_state<true>, its counters and its progress -- is
// published to the next warp by the release store of the ring entry (no separate fence): the other
// lanes' stores are ordered before it by __syncwarp (cumulativity), and the next warp's acquire load
// of the entry, followed by __syncwarp, orders all its lanes' loads after it.  A unit sits in the ring
// at most once, so one warp at a time owns it and read-modify-writes of its state need no atomics.
template <class Body>
__device__ __forceinline__ void sched_serve(long long *sched, long long n_units, long long n_steps, int chunk, int lane,
                                            const Body &body) {
    const SchedView Q(sched, n_units);
    const unsigned long long cap = (unsigned long long)Q.cap;
    const long long items_per_unit = (n_steps + chunk - 1) / chunk;
    const unsigned long long total = (unsigned long long)n_units * (unsigned long long)items_per_unit;
    while (true) {
        PROF_T(t0);
        unsigned long long idx = 0;
        if (lane == 0) idx = atomicAdd(Q.head, 1ull);
        idx = __shfl_sync(FULL, idx, 0);
        if (idx >= total) break;
        unsigned long long *slot = Q.ring + idx % cap;
        const unsigned long long want = idx / cap + 1;
        const unsigned long long e = spin_until(slot, lane, [want](unsigned long long v) { return (v >> 32) == want; });
        // mark the slot consumed: ordered after our own read of it (same address), nothing to publish
        if (lane == 0) st_relaxed_u64(slot, 0ull);
        __syncwarp();
        const long long unit = (long long)(e & 0xffffffffull);
        const long long s0 = __ldcg(Q.progress + unit);
        const long long s1 = (s0 + chunk < n_steps) ? s0 + chunk : n_steps;
        PROF_T(t1);
        body(unit, s0, s1);
        PROF_T(t2);
        if (lane == 0) __stcg(Q.progress + unit, s1);
        __syncwarp();
        if (s1 < n_steps) {   // warp-uniform
            unsigned long long t = 0;
            if (lane == 0) t = atomicAdd(Q.tail, 1ull);
            t = __shfl_sync(FULL, t, 0);
            unsigned long long *pslot = Q.ring + t % cap;
            spin_until(pslot, lane, [](unsigned long long v) { return v == 0ull; });   // previous lap consumed (cap = 2n: no wait in practice)
            if (lane == 0) st_release_u64(pslot, ((t / cap + 1) << 32) | (unsigned long long)unit);
        }
        __syncwarp();
        PROF_T(t3);
        PROF_ADD(0, t0, t3);
        PROF_ADD(1, t0, t1);
        PROF_ADD(6, t1, t2);
        PROF_ADD(7, t2, t3);
        PROF_ADD(8, 0, 1);
    }
}

}  // namespace ipmcmc
