// Kernels of a user-written CUDA model (BK_MODEL_USER_CUDA, bk.h).  The host side (user_model.cu) includes this file
// for UserRunArgs only; the kernels are compiled at run time by NVRTC, one library per (source, D, dtype), from
//   integer typedefs + device_rng.cuh + `typedef float|double bk_real;` + the user's source + this file
// with -DBK_DIMS=D.  The user's source defines
//   __device__ bk_real log_density_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
//
// bk_user_eval      one thread per chain on global rows: model_eval's case for this kind, through which the
//                   generic HMC / MALA / RW-Metropolis engine, the lockstep DrGHMC engine and the Stretcher run.
// bk_user_hmc/mala/mh
//                   fused samplers, one thread per chain: theta, its gradient and log density stay in registers
//                   across all n_draws of a call.  Randomness and arithmetic follow the generic engine exactly
//                   (Row<T> and k_hmc_* / k_mala_* / k_mh_* in sampler_generic.cu): philox_normal4 per block of 4
//                   elements, philox_accept_uniform at block ceil(D / 4), the same sequence of Ar<T> operations;
//                   in fp64 only the summation order of the kinetic / proposal-energy sums differs.
#pragma once

namespace bk {

// Launch arguments of bk_user_hmc / bk_user_mala / bk_user_mh.  Plain fields only: the host (nvcc) and the kernels
// (NVRTC) must agree on the layout.  Pointers are in the model's dtype unless typed.
struct UserRunArgs {
    void* theta;              // [C, D] in/out
    const void* params;       // [n_params] or NULL
    const void* metric;       // HMC: [D] or NULL (identity)
    const void* normals;      // injected [n, C, D] or NULL (Philox)
    const void* uniforms;     // injected [n, C, n_uniform]
    void* draws;              // [n, C, D] or NULL
    void* logp;               // [n, C] or NULL
    int32_t* accept;          // [n, C] or NULL
    int64_t C, n_draws;
    uint64_t seed, draw_offset, chain_offset;
    int32_t rng_mode, n_uniform;
    int32_t L, hastings;
    double eps, half_eps;     // HMC; MALA: eps
    double sd, coef;          // MALA: sqrt(2 eps), -0.25 / eps
    double scale, s2;         // RW-Metropolis
};

}  // namespace bk

#ifdef __CUDACC_RTC__

namespace bk {
namespace user {

constexpr int D = BK_DIMS;
constexpr int NB = (D + 3) / 4;   // element blocks of 4
using T = bk_real;
using A = Ar<T>;

// normals of element block b of (chain c, draw t): the rule of Row<T>::normal4
__device__ __forceinline__ void normal4(const UserRunArgs& a, int64_t c, int64_t t, int b, T (&z)[4]) {
    if (a.rng_mode == 1) {   // BK_RNG_INJECTED
        const T* p = reinterpret_cast<const T*>(a.normals) + (t * a.C + c) * (int64_t)D;
#pragma unroll
        for (int i = 0; i < 4; ++i) z[i] = (4 * b + i < D) ? p[4 * b + i] : T(0);
    } else {
        philox_normal4<T>(a.seed, (uint32_t)b, (uint32_t)(a.chain_offset + (uint64_t)c),
                          (uint32_t)(a.draw_offset + (uint64_t)t), z);
    }
}

// the accept uniform: Row<T>::uniform(0)
__device__ __forceinline__ T accept_uniform(const UserRunArgs& a, int64_t c, int64_t t) {
    if (a.rng_mode == 1) return reinterpret_cast<const T*>(a.uniforms)[(t * a.C + c) * a.n_uniform];
    if (a.n_uniform == 1)
        return philox_accept_uniform<T>(a.seed, (uint32_t)(a.chain_offset + (uint64_t)c),
                                        (uint32_t)(a.draw_offset + (uint64_t)t), D);
    return philox_uniform<T>(a.seed, 0u, (uint32_t)(a.chain_offset + (uint64_t)c),
                             (uint32_t)(a.draw_offset + (uint64_t)t));
}

// all D normals of (c, t)
__device__ __forceinline__ void normals(const UserRunArgs& a, int64_t c, int64_t t, T (&z)[D]) {
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        T z4[4];
        normal4(a, c, t, b, z4);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (4 * b + i < D) z[4 * b + i] = z4[i];
    }
}

__device__ __forceinline__ void load_row(const T* p, T (&v)[D]) {
#pragma unroll
    for (int e = 0; e < D; ++e) v[e] = p[e];
}

__device__ __forceinline__ void emit(const UserRunArgs& a, int64_t c, int64_t t, const T (&th)[D], T lp, bool acc) {
    if (a.draws) {
        T* dr = reinterpret_cast<T*>(a.draws) + (t * a.C + c) * (int64_t)D;
#pragma unroll
        for (int e = 0; e < D; ++e) dr[e] = th[e];
    }
    if (a.logp) reinterpret_cast<T*>(a.logp)[t * a.C + c] = lp;
    if (a.accept) a.accept[t * a.C + c] = acc ? 1 : 0;
}

}  // namespace user
}  // namespace bk

// theta [C, D] -> lp [C] (nullable), grad [C, D]
extern "C" __global__ void __launch_bounds__(128) bk_user_eval(const bk_real* __restrict__ theta, long long C,
                                                               const bk_real* __restrict__ params,
                                                               bk_real* __restrict__ lp, bk_real* __restrict__ grad) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const bk_real v = log_density_gradient(theta + c * BK_DIMS, grad + c * BK_DIMS, params);
    if (lp) lp[c] = v;
}

// The fused samplers are compiled only where the library dispatches to them (D <= BK_USER_FUSED_MAX_D).
#if BK_DIMS <= BK_USER_FUSED_MAX_D

// HMCDiag: k_hmc_begin / k_hmc_step / k_hmc_end with the state in registers
extern "C" __global__ void __launch_bounds__(128) bk_user_hmc(const bk::UserRunArgs a) {
    using namespace bk::user;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.C) return;
    const T* params = reinterpret_cast<const T*>(a.params);
    const T* metric = reinterpret_cast<const T*>(a.metric);
    const T eps = (T)a.eps, half_eps = (T)a.half_eps;
    T* row = reinterpret_cast<T*>(a.theta) + c * (int64_t)D;
    T th[D], g[D];
    load_row(row, th);
    T lp = log_density_gradient(th, g, params);
    for (int64_t t = 0; t < a.n_draws; ++t) {
        T q[D], r[D], gq[D];
        normals(a, c, t, r);
        T kin = T(0);
#pragma unroll
        for (int e = 0; e < D; ++e) {
            const T z = r[e];
            const T m = metric ? metric[e] : T(1);
            const T mg = metric ? A::mul(m, g[e]) : g[e];
            kin = A::add(kin, A::mul(z, metric ? A::mul(m, z) : z));
            T re = A::sub(z, A::mul(half_eps, mg));
            T qe = th[e];
            if (a.L > 0) {
                re = A::add(re, A::mul(eps, mg));
                qe = A::add(qe, A::mul(eps, re));
            }
            r[e] = re;
            q[e] = qe;
        }
        const T h0 = A::sub(lp, A::mul(T(0.5), kin));
        T lpq = lp;
#pragma unroll
        for (int e = 0; e < D; ++e) gq[e] = g[e];
        for (int s = 0; s < a.L; ++s) {
            lpq = log_density_gradient(q, gq, params);
            if (s + 1 < a.L) {
#pragma unroll
                for (int e = 0; e < D; ++e) {
                    const T mg = metric ? A::mul(metric[e], gq[e]) : gq[e];
                    r[e] = A::add(r[e], A::mul(eps, mg));
                    q[e] = A::add(q[e], A::mul(eps, r[e]));
                }
            }
        }
        kin = T(0);
#pragma unroll
        for (int e = 0; e < D; ++e) {
            const T m = metric ? metric[e] : T(1);
            const T mg = metric ? A::mul(m, gq[e]) : gq[e];
            const T re = A::add(r[e], A::mul(half_eps, mg));
            kin = A::add(kin, A::mul(re, metric ? A::mul(m, re) : re));
        }
        const T h1 = A::sub(lpq, A::mul(T(0.5), kin));
        const bool acc = bk::log_u(accept_uniform(a, c, t)) < A::sub(h1, h0);
        if (acc) {
#pragma unroll
            for (int e = 0; e < D; ++e) {
                th[e] = q[e];
                g[e] = gq[e];
            }
            lp = lpq;
        }
        emit(a, c, t, th, acc ? h1 : h0, acc);
    }
#pragma unroll
    for (int e = 0; e < D; ++e) row[e] = th[e];
}

// MALA: k_mala_propose / k_mala_accept
extern "C" __global__ void __launch_bounds__(128) bk_user_mala(const bk::UserRunArgs a) {
    using namespace bk::user;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.C) return;
    const T* params = reinterpret_cast<const T*>(a.params);
    const T eps = (T)a.eps, sd = (T)a.sd, coef = (T)a.coef;
    T* row = reinterpret_cast<T*>(a.theta) + c * (int64_t)D;
    T th[D], g[D];
    load_row(row, th);
    T lp = log_density_gradient(th, g, params);
    for (int64_t t = 0; t < a.n_draws; ++t) {
        T q[D], gq[D];
        normals(a, c, t, q);
#pragma unroll
        for (int e = 0; e < D; ++e) q[e] = A::add(A::add(th[e], A::mul(eps, g[e])), A::mul(sd, q[e]));
        const T lpq = log_density_gradient(q, gq, params);
        T sf = T(0), sr = T(0);
#pragma unroll
        for (int e = 0; e < D; ++e) {
            const T df = A::sub(A::sub(q[e], th[e]), A::mul(eps, g[e]));
            const T dr = A::sub(A::sub(th[e], q[e]), A::mul(eps, gq[e]));
            sf = A::add(sf, A::mul(df, df));
            sr = A::add(sr, A::mul(dr, dr));
        }
        const T fwd = A::mul(coef, sf), rev = A::mul(coef, sr);
        const bool acc = bk::log_u(accept_uniform(a, c, t)) < A::add(A::sub(lpq, lp), A::sub(rev, fwd));
        if (acc) {
#pragma unroll
            for (int e = 0; e < D; ++e) {
                th[e] = q[e];
                g[e] = gq[e];
            }
            lp = lpq;
        }
        emit(a, c, t, th, lp, acc);
    }
#pragma unroll
    for (int e = 0; e < D; ++e) row[e] = th[e];
}

// Metropolis / MetropolisHastings with the Gaussian random walk: k_mh_propose / k_mh_accept.  The gradient the
// user's function writes is never read: after inlining its computation is dead code.
extern "C" __global__ void __launch_bounds__(128) bk_user_mh(const bk::UserRunArgs a) {
    using namespace bk::user;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.C) return;
    const T* params = reinterpret_cast<const T*>(a.params);
    const T scale = (T)a.scale, s2 = (T)a.s2;
    T* row = reinterpret_cast<T*>(a.theta) + c * (int64_t)D;
    T th[D], unused[D];
    load_row(row, th);
    T lp = log_density_gradient(th, unused, params);
    for (int64_t t = 0; t < a.n_draws; ++t) {
        T q[D];
        normals(a, c, t, q);
#pragma unroll
        for (int e = 0; e < D; ++e) q[e] = A::add(th[e], A::mul(scale, q[e]));
        const T lpq = log_density_gradient(q, unused, params);
        T ratio = A::sub(lpq, lp);
        if (a.hastings) {
            T sf = T(0), sr = T(0);
#pragma unroll
            for (int e = 0; e < D; ++e) {
                const T df = A::sub(q[e], th[e]), dr = A::sub(th[e], q[e]);
                sf = A::add(sf, A::mul(df, df));
                sr = A::add(sr, A::mul(dr, dr));
            }
            const T fwd = A::mul(T(-0.5), sf) / s2, rev = A::mul(T(-0.5), sr) / s2;
            ratio = A::add(ratio, A::sub(rev, fwd));
        }
        const bool acc = bk::log_u(accept_uniform(a, c, t)) < ratio;
        if (acc) {
#pragma unroll
            for (int e = 0; e < D; ++e) th[e] = q[e];
            lp = lpq;
        }
        emit(a, c, t, th, lp, acc);
    }
#pragma unroll
    for (int e = 0; e < D; ++e) row[e] = th[e];
}

#endif  // BK_DIMS <= BK_USER_FUSED_MAX_D
#endif  // __CUDACC_RTC__
