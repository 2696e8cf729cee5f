// Device-only arithmetic and random streams shared by nvcc and NVRTC: the strict arithmetic traits (fp64 parity
// mode), Philox4x32-10, the fast Box-Muller, the uniform grids and the accept-uniform rule of the single-uniform
// samplers.  The library's kernels get it through common.cuh; a runtime-compiled user model (user_model.cu) gets the
// same text embedded in the library, so its chains consume the same Philox words as the built-in plugins' chains.
// NVRTC has no standard headers: under it the includer defines the fixed-width integer typedefs first.
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>
#endif

namespace bk {
// ---- arithmetic traits -------------------------------------------------------
// fp64 = parity mode: NumPy performs separate multiply and add roundings, so
// contraction into FMA is forbidden (SURVEY.md 2.1-5).  fp32 = timed mode: the
// compiler is free to contract.
template <typename T>
struct Ar;
template <>
struct Ar<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
    static __device__ __forceinline__ float sub(float a, float b) { return a - b; }
    static __device__ __forceinline__ float log_(float a) { return logf(a); }
    static __device__ __forceinline__ float exp_(float a) { return expf(a); }
    static __device__ __forceinline__ float sqrt_(float a) { return sqrtf(a); }
    static __device__ __forceinline__ float log1p_(float a) { return log1pf(a); }
};
template <>
struct Ar<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
    static __device__ __forceinline__ double log_(double a) { return log(a); }
    static __device__ __forceinline__ double exp_(double a) { return exp(a); }
    static __device__ __forceinline__ double sqrt_(double a) { return sqrt(a); }
    static __device__ __forceinline__ double log1p_(double a) { return log1p(a); }
};

template <typename T>
__device__ __forceinline__ T neg_inf() {
    return -__int_as_float(0x7f800000);
}

// ---- Philox4x32-10 -----------------------------------------------------------
struct Philox {
    static constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    static constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    static __host__ __device__ __forceinline__ void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
        uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
#else
        uint64_t p0 = (uint64_t)M0 * c[0], p1 = (uint64_t)M1 * c[2];
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
        uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
        uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    }
    // counter = (block, tag, chain, draw), key = seed
    static __host__ __device__ __forceinline__ void gen(uint64_t seed, uint32_t block, uint32_t tag,
                                                        uint32_t chain, uint32_t draw,
                                                        uint32_t (&out)[4]) {
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
        out[0] = block; out[1] = tag; out[2] = chain; out[3] = draw;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            round(out, k0, k1);
            k0 += W0; k1 += W1;
        }
    }
};

// tags separate the independent streams of one (chain, draw)
enum : uint32_t { TAG_NORMAL = 0, TAG_NORMAL_HI = 1, TAG_UNIFORM = 2, TAG_RESAMPLE = 3 };

// uniforms strictly inside (0,1): midpoints of the 2^-23 / 2^-52 grid.  k + 0.5 must be REPRESENTABLE (24 / 53
// significant bits), otherwise round-to-even turns the top of the range into exactly 1.0: 23 / 52 random bits.
__host__ __device__ __forceinline__ float u01(uint32_t x) { return ((x >> 9) + 0.5f) * 1.1920928955078125e-7f; }
__host__ __device__ __forceinline__ double u01d(uint32_t hi, uint32_t lo) {
    return (((double)(hi >> 6)) * 67108864.0 + (double)(lo >> 6) + 0.5) * 2.220446049250313e-16;
}

// Box-Muller on the SFU, fp32, straight from the counter-mode words (no intermediate u01 grid): ~6 instructions per
// normal.  Radius: u = (w + 0.5) 2^-32 rounded to fp32, in (0, 1] (2^-33 at w = 0: |z| <= 6.8; exactly 1 with
// probability 2^-25: radius 0), r = sqrt(-2 ln u) by lg2.approx / sqrt.approx (u is never denormal, so none of the
// range fix-ups of logf / sqrtf are needed).  Angle: the word read as a SIGNED integer times 2 pi / 2^32, i.e. already
// folded into [-pi, pi], where sin.approx / cos.approx have ~2^-21 absolute error -- far below fp32 sampling noise.
__device__ __forceinline__ float bm_radius(uint32_t w) {
    const float u = fmaf(__uint2float_rn(w), 2.3283064365386963e-10f, 1.1641532182693481e-10f);
    float l, r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(u));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(l * -1.3862943611198906f));
    return r;
}
__device__ __forceinline__ void bm_sincos(uint32_t w, float& s, float& c) {
    const float a = __int2float_rn((int32_t)w) * 1.4629180792671596e-9f;
    asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(a));
    asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c) : "f"(a));
}
__device__ __forceinline__ void box_muller4(const uint32_t (&r)[4], float (&z)[4]) {
    const float r0 = bm_radius(r[0]), r1 = bm_radius(r[2]);
    float s0, c0, s1, c1;
    bm_sincos(r[1], s0, c0);
    bm_sincos(r[3], s1, c1);
    z[0] = r0 * c0; z[1] = r0 * s0; z[2] = r1 * c1; z[3] = r1 * s1;
}

// 4 standard normals for element block `block` of (chain, draw)
// (raw2, when given, receives the first two counter-mode words of the block: a caller whose block
// holds no valid element may spend them on something else, e.g. an accept uniform)
template <typename T>
__device__ __forceinline__ void philox_normal4(uint64_t seed, uint32_t block, uint32_t chain,
                                               uint32_t draw, T (&z)[4], uint32_t* raw2 = nullptr);
template <>
__device__ __forceinline__ void philox_normal4<float>(uint64_t seed, uint32_t block, uint32_t chain,
                                                      uint32_t draw, float (&z)[4], uint32_t* raw2) {
    uint32_t r[4];
    Philox::gen(seed, block, TAG_NORMAL, chain, draw, r);
    if (raw2) { raw2[0] = r[0]; raw2[1] = r[1]; }
    box_muller4(r, z);
}
template <>
__device__ __forceinline__ void philox_normal4<double>(uint64_t seed, uint32_t block, uint32_t chain,
                                                       uint32_t draw, double (&z)[4], uint32_t* raw2) {
    uint32_t a[4], b[4];
    Philox::gen(seed, block, TAG_NORMAL, chain, draw, a);
    if (raw2) { raw2[0] = a[0]; raw2[1] = a[1]; }
    Philox::gen(seed, block, TAG_NORMAL_HI, chain, draw, b);
    double r0 = sqrt(-2.0 * log(u01d(a[0], a[1]))), r1 = sqrt(-2.0 * log(u01d(b[0], b[1])));
    double s0, c0, s1, c1;
    sincospi(2.0 * u01d(a[2], a[3]), &s0, &c0);
    sincospi(2.0 * u01d(b[2], b[3]), &s1, &c1);
    z[0] = r0 * c0; z[1] = r0 * s0; z[2] = r1 * c1; z[3] = r1 * s1;
}

// k-th uniform of (chain, draw)
// (boff: added to the block counter word -- move j of an SMC temperature step draws at boff = 2^16 j, smc_move_block)
template <typename T>
__host__ __device__ __forceinline__ T philox_uniform(uint64_t seed, uint32_t k, uint32_t chain, uint32_t draw,
                                                     uint32_t tag = TAG_UNIFORM, uint32_t boff = 0);
template <>
__host__ __device__ __forceinline__ float philox_uniform<float>(uint64_t seed, uint32_t k, uint32_t chain,
                                                                uint32_t draw, uint32_t tag, uint32_t boff) {
    uint32_t r[4];
    Philox::gen(seed, (k >> 2) + boff, tag, chain, draw, r);
    return u01(r[k & 3]);
}
template <>
__host__ __device__ __forceinline__ double philox_uniform<double>(uint64_t seed, uint32_t k, uint32_t chain,
                                                                  uint32_t draw, uint32_t tag, uint32_t boff) {
    uint32_t r[4];
    Philox::gen(seed, (k >> 1) + boff, tag, chain, draw, r);
    return (k & 1) ? u01d(r[2], r[3]) : u01d(r[0], r[1]);
}

// Accept uniform of the single-uniform samplers (HMC / MALA / RW-Metropolis) in Philox mode: the first words of
// element block B = ceil(D / 4) of the NORMAL stream -- the first block no element of the proposal uses.  A fused
// register-resident kernel whose lane layout has a slot for block B gets it from the pass that makes the normals
// (one counter-mode call per lane and draw instead of two); every other engine makes one extra call.  The rule
// does not depend on the layout, so chains do not depend on which engine (or lane layout) ran.
__host__ __device__ __forceinline__ int accept_block(int D) { return (D + 3) >> 2; }
template <typename T>
__device__ __forceinline__ T uniform_of_words(uint32_t w0, uint32_t w1) {
    if constexpr (sizeof(T) == 4) return u01(w0);
    else return u01d(w0, w1);
}
template <typename T>
__device__ __forceinline__ T philox_accept_uniform(uint64_t seed, uint32_t chain, uint32_t draw, int D, uint32_t boff = 0) {
    uint32_t r[4];
    Philox::gen(seed, (uint32_t)accept_block(D) + boff, TAG_NORMAL, chain, draw, r);
    return uniform_of_words<T>(r[0], r[1]);
}

// Several Markov moves per SMC temperature step (bk_smc_kernel.moves): move j draws exactly the words move 0 draws
// (normals, accept uniform, fp64 TAG_NORMAL_HI words, a proposal's TAG_UNIFORM uniforms) with the element-block counter
// word b replaced by b + 2^16 j.  Every block a move uses is below 2^16 (D <= 256, <= 512 proposal normals, <= 64
// uniforms), so move 0 is the single-move stream and the moves' streams are disjoint.
__host__ __device__ __forceinline__ uint32_t smc_move_block(int j) { return (uint32_t)j << 16; }

// Normals of a user proposal (bk_proposal_create_cuda): normal k is element k % 4 of philox_normal4 on element block
// proposal_normal_block(k, D) -- the blocks 0, 1, ... with accept_block(D) skipped, so the accept uniform never shares
// its words with a proposal normal, and a proposal with at most D normals reads exactly the random walk's normals.
__host__ __device__ __forceinline__ int proposal_normal_block(int k, int D) {
    const int b = k >> 2;
    return b < accept_block(D) ? b : b + 1;
}

// log(u) with numpy semantics for u == 0 (-inf: always accepts)
template <typename T>
__device__ __forceinline__ T log_u(T u) {
    return u > T(0) ? Ar<T>::log_(u) : neg_inf<T>();
}

}  // namespace bk
