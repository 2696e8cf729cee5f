// Shared device/host helpers for libbk_b200: error plumbing, group reductions; the strict arithmetic traits
// (fp64 parity mode) and Philox4x32-10 come from device_rng.cuh.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>

#include "../../include/bk.h"
#include "device_rng.cuh"

namespace bk {

// ---- host-side error plumbing ---------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
inline void count_launch(uint64_t n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define BK_CHECK_ARG(cond, ...)                 \
    do {                                        \
        if (!(cond)) {                          \
            bk::set_error(__VA_ARGS__);         \
            return BK_E_INVALID;                \
        }                                       \
    } while (0)

#define BK_CUDA(call)                                                                   \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            bk::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),      \
                          __FILE__, __LINE__);                                          \
            return BK_E_CUDA;                                                           \
        }                                                                               \
    } while (0)

#define BK_LAUNCH_CHECK()                                                               \
    do {                                                                                \
        bk::count_launch();                                                             \
        cudaError_t e_ = cudaGetLastError();                                            \
        if (e_ != cudaSuccess) {                                                        \
            bk::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_),  \
                          __FILE__, __LINE__);                                          \
            return BK_E_CUDA;                                                           \
        }                                                                               \
    } while (0)

// optional event timing of selected launches (see bk_profile_* in bk.h)
void prof_begin(int tag, cudaStream_t st);
void prof_end(int tag, cudaStream_t st);

// BK_FORCE_GENERIC=1 routes every model through the generic engines (test hook: both engines must produce the same
// chains)
bool force_generic();

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocator over the caller-provided workspace
struct Arena {
    char* base;
    size_t cap, off;
    Arena(void* p, size_t n) : base((char*)p), cap(n), off(0) {}
    template <typename T>
    T* take(size_t n) {
        off = align_up(off, 256);
        T* r = (T*)(base + off);
        off += n * sizeof(T);
        return r;
    }
    bool ok() const { return off <= cap && (base != nullptr || off == 0); }
};

// ---- reductions over a group of G consecutive lanes (G power of two <= 32) ---
template <int G, typename T>
__device__ __forceinline__ T group_sum(T v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_sum(T v) { return group_sum<32, T>(v); }
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// block-wide sum for blockDim.x <= 1024 (result valid in every thread)
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem /*>=33*/) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) smem[w] = v;
    __syncthreads();
    if (w == 0) {
        T t = lane < nw ? smem[lane] : T(0);
        t = warp_sum(t);
        if (lane == 0) smem[32] = t;
    }
    __syncthreads();
    return smem[32];
}

template <typename T>
struct DType;
template <>
struct DType<float> { static constexpr int id = BK_F32; };
template <>
struct DType<double> { static constexpr int id = BK_F64; };

}  // namespace bk
