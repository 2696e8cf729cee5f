// Device side of the sharded particle system's cross-rank protocol (smc_shard.cuh): the shard geometry, the mailbox
// layout, the acquire / release helpers, the bounded wait and the posts.  Shared by nvcc and NVRTC: the library's SMC
// kernels get it through smc_shard.cuh; the SMC kernels of a runtime-compiled user model (user_kernels.cuh) get the
// same text embedded in the library, so both talk the same protocol.  Under NVRTC the includer defines the fixed-width
// integer typedefs and BK_SMC_MAX_WORLD / BK_SMC_MAILBOX_BYTES (from bk.h's values) first.
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bk.h"
#endif

namespace bk {

struct ShardGeom {
    int32_t world, rank;   // world == 0: not a sharded call
    int32_t extra, small;  // first `extra` ranks hold base + 1 items; small: every id fits 32 bits
    int64_t M, base;       // global item count, floor(M / world)
};

__host__ __device__ __forceinline__ int64_t shard_lo(const ShardGeom& g, int r) {
    return (int64_t)r * g.base + (r < g.extra ? r : g.extra);
}
__host__ __device__ __forceinline__ int64_t shard_n(const ShardGeom& g, int r) { return g.base + (r < g.extra ? 1 : 0); }

// owner rank and local row of global id gid
__device__ __forceinline__ void shard_locate(const ShardGeom& g, int64_t gid, int& r, int64_t& loc) {
    const int64_t cut = (int64_t)g.extra * (g.base + 1);
    if (g.small) {
        const uint32_t u = (uint32_t)gid, c = (uint32_t)cut;
        if (u < c) { const uint32_t q = u / (uint32_t)(g.base + 1); r = (int)q; loc = u - q * (uint32_t)(g.base + 1); }
        else { const uint32_t q = (u - c) / (uint32_t)g.base; r = g.extra + (int)q; loc = (u - c) - q * (uint32_t)g.base; }
    } else {
        if (gid < cut) { const int64_t q = gid / (g.base + 1); r = (int)q; loc = gid - q * (g.base + 1); }
        else { const int64_t q = (gid - cut) / g.base; r = g.extra + (int)q; loc = (gid - cut) - q * g.base; }
    }
}

// ---- mailbox layout (64-bit words; one mailbox per rank, written by every rank) -----------------
// word 0: error word (0 = fine; 1 = a wait timed out; 2 = all weights vanished)
// slots are indexed [parity of the step][source rank]
enum : int {
    MB_ERR = 0,
    MB_MAX = 8,                                   // {max (double bits), step}
    MB_MASS = MB_MAX + 2 * BK_SMC_MAX_WORLD * 2,  // {W (int64), Q (double bits), n_local, step}
    MB_DONE = MB_MASS + 2 * BK_SMC_MAX_WORLD * 4, // {step}
    MB_WORDS = MB_DONE + 2 * BK_SMC_MAX_WORLD
};
static_assert(MB_WORDS * 8 <= BK_SMC_MAILBOX_BYTES, "mailbox size");

__device__ __forceinline__ void st_release_sys(uint64_t* p, uint64_t v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t ld_relaxed_sys(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t ld_relaxed_gpu(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu(uint64_t* p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_gpu_f64(const double* p) {
    return __longlong_as_double((long long)ld_relaxed_gpu(reinterpret_cast<const uint64_t*>(p)));
}
__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Wait until the step word at `flag` (in OUR mailbox) reaches `step`.  Bounded: a rank that never
// arrives (crashed peer) makes the wait give up after BK_SMC_WAIT_NS, flags the error word and lets the
// kernel run to completion on garbage -- the host raises when it next looks at the mailbox.
constexpr uint64_t BK_SMC_WAIT_NS = 20ull * 1000 * 1000 * 1000;
__device__ __forceinline__ bool mail_wait(const uint64_t* flag, uint64_t step, uint64_t* mailbox) {
    if (ld_acquire_sys(flag) >= step) return true;
    if (ld_relaxed_sys(mailbox + MB_ERR) == 1ull) return false;   // a wait already timed out: the run is lost, do not wait again
    const uint64_t t0 = global_ns();
    unsigned it = 0;
    while (ld_acquire_sys(flag) < step) {
        __nanosleep(64);
        if ((++it & 1023u) == 0 && global_ns() - t0 > BK_SMC_WAIT_NS) {
            st_relaxed_sys(mailbox + MB_ERR, 1ull);
            return false;
        }
    }
    return true;
}
// post {payload, step} / {p0, p1, p2, step}: payload first, then a release store of the step number
__device__ __forceinline__ void mail_post1(uint64_t* slot, uint64_t payload, uint64_t step) {
    st_relaxed_sys(slot, payload);
    st_release_sys(slot + 1, step);
}
__device__ __forceinline__ void mail_post3(uint64_t* slot, uint64_t p0, uint64_t p1, uint64_t p2, uint64_t step) {
    st_relaxed_sys(slot, p0);
    st_relaxed_sys(slot + 1, p1);
    st_relaxed_sys(slot + 2, p2);
    st_release_sys(slot + 3, step);
}

constexpr int SMC_MAXPART = 2048;   // per-CTA partials of a move kernel's statistics epilogue (its grid is capped there)

// Statistics epilogue of a move kernel: the local maximum of the log-weights leaves with the launch -- every CTA
// stores its maximum into maxpart[blockIdx.x], the last CTA to finish (ticket) reduces them and posts (max, epoch)
// into every rank's mailbox.  Called by every thread of every CTA; blockDim.x is a multiple of 32.  The user-model
// kernels call it; k_smc_move_weight (smc.cu) keeps its own inline copy of the same steps, because calling this
// function there changes that kernel's register allocation.
__device__ __forceinline__ double warp_max_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ void smc_post_max(double lw_max, double* maxpart, unsigned* ticket, const ShardGeom& sh,
                                             uint64_t* const* mail_tab, uint64_t epoch) {
    __shared__ double red[33];
    __shared__ bool last_s;
    double v = warp_max_f64(lw_max);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) red[w] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) v = fmax(v, red[i]);
        maxpart[blockIdx.x] = v;
        __threadfence();
        last_s = atomicInc(ticket, gridDim.x - 1) == gridDim.x - 1;   // wraps to 0: self-resetting
    }
    __syncthreads();
    if (last_s) {
        __threadfence();
        double m2 = -__longlong_as_double(0x7ff0000000000000ll);   // -inf
        for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) m2 = fmax(m2, ld_relaxed_gpu_f64(maxpart + i));
        m2 = warp_max_f64(m2);
        __syncthreads();
        if (lane == 0) red[w] = m2;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m2 = fmax(m2, red[i]);
            red[32] = m2;
        }
        __syncthreads();
        const int nw = sh.world > 0 ? sh.world : 1;
        if ((int)threadIdx.x < nw)
            mail_post1(mail_tab[threadIdx.x] + MB_MAX + ((epoch & 1) * BK_SMC_MAX_WORLD + sh.rank) * 2,
                       (uint64_t)__double_as_longlong(red[32]), epoch);
    }
}

}  // namespace bk
