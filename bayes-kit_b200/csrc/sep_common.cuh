// Register-resident chain state for the fused "separable model" samplers.
//
// A chain is owned by a group of G consecutive lanes (G = 1..32); each lane
// keeps NE = 4*J elements of every per-dimension vector in registers:
// element e = 4*(lane + G*j) + i  (j < J, i < 4), i.e. float4-vectorised,
// lane-strided -> every global access of a group is one contiguous segment.
// theta / rho never touch HBM between the L leapfrog steps of a draw.
#pragma once
#include "common.cuh"

namespace bk {

enum { MK_ISO = 0, MK_DIAG = 1 };

template <typename T>
struct SepModel {
    const T* mu;      // [D] or NULL
    const T* prec;    // [D] or NULL (-> prec_scalar)
    T prec_scalar;
    const T* metric;  // [D] or NULL (identity)
};

// VM fixes the row access mode at compile time (hot kernels: no per-block path selection in the instruction stream):
// -1 = decided at run time by vec / vec2, 0 = scalar, 1 = 128-bit (D % 4 == 0, rows 16-byte aligned), 2 = 64-bit
// (fp32, D even, rows 8-byte aligned).
template <typename T, int G, int J, int VM = -1>
struct Lanes {
    static constexpr int NE = 4 * J;
    int lane;   // lane within group
    int D;
    bool vec;
    bool vec2 = false;   // fp32, D even, rows 8-byte aligned (e.g. D = 50): 64-bit accesses, two per element block
    __device__ __forceinline__ bool m_vec() const { return VM < 0 ? vec : VM == 1; }
    __device__ __forceinline__ bool m_vec2() const { return VM < 0 ? (sizeof(T) == 4 && vec2) : (sizeof(T) == 4 && VM == 2); }
    __device__ __forceinline__ int elem(int k) const { return 4 * (lane + G * (k >> 2)) + (k & 3); }
    __device__ __forceinline__ bool valid(int k) const { return elem(k) < D; }

    __device__ __forceinline__ void load(const T* row, T (&v)[NE], T fill) const {
#pragma unroll
        for (int j = 0; j < J; ++j) {
            int e0 = 4 * (lane + G * j);
            if (VM == 1 && e0 >= D) {   // D % 4 == 0: a block is all valid or all padding
#pragma unroll
                for (int i = 0; i < 4; ++i) v[4 * j + i] = fill;
            } else if (VM == 1 || (m_vec() && e0 + 3 < D)) {
                if constexpr (sizeof(T) == 4) {
                    float4 t = *reinterpret_cast<const float4*>(row + e0);
                    v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
                } else {
                    double2 a = *reinterpret_cast<const double2*>(row + e0);
                    double2 b = *reinterpret_cast<const double2*>(row + e0 + 2);
                    v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = b.x; v[4 * j + 3] = b.y;
                }
            } else if (m_vec2()) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (e0 + 2 * h + 1 < D) {
                        const float2 t = *reinterpret_cast<const float2*>(row + e0 + 2 * h);
                        v[4 * j + 2 * h] = t.x; v[4 * j + 2 * h + 1] = t.y;
                    } else {
                        v[4 * j + 2 * h] = fill; v[4 * j + 2 * h + 1] = fill;
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) v[4 * j + i] = (e0 + i < D) ? row[e0 + i] : fill;
            }
        }
    }
    __device__ __forceinline__ void store(T* row, const T (&v)[NE]) const {
#pragma unroll
        for (int j = 0; j < J; ++j) {
            int e0 = 4 * (lane + G * j);
            if (VM == 1 && e0 >= D) {
            } else if (VM == 1 || (m_vec() && e0 + 3 < D)) {
                if constexpr (sizeof(T) == 4) {
                    *reinterpret_cast<float4*>(row + e0) =
                        make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                } else {
                    *reinterpret_cast<double2*>(row + e0) = make_double2(v[4 * j], v[4 * j + 1]);
                    *reinterpret_cast<double2*>(row + e0 + 2) = make_double2(v[4 * j + 2], v[4 * j + 3]);
                }
            } else if (m_vec2()) {
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (e0 + 2 * h + 1 < D)
                        *reinterpret_cast<float2*>(row + e0 + 2 * h) = make_float2(v[4 * j + 2 * h], v[4 * j + 2 * h + 1]);
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (e0 + i < D) row[e0 + i] = v[4 * j + i];
            }
        }
    }
    // standard normals for (chain, draw); invalid slots are 0
    // raw2 (optional): the first two Philox words of element block `ub`, left in the lane that owns that block
    // (lane ub % G) -- the accept uniform of common.cuh's rule when the layout has a slot for it (ub < G * J)
    __device__ __forceinline__ void normals(const bk_rng& rng, int64_t C, int64_t chain, int64_t t,
                                            T (&z)[NE], uint32_t* raw2 = nullptr, int ub = -1) const {
        if (rng.mode == BK_RNG_INJECTED) {
            load(reinterpret_cast<const T*>(rng.normals) + (t * C + chain) * (int64_t)D, z, T(0));
        } else {
            uint32_t gc = (uint32_t)(rng.chain_offset + (uint64_t)chain);
            uint32_t gd = (uint32_t)(rng.draw_offset + (uint64_t)t);
#pragma unroll
            for (int j = 0; j < J; ++j) {
                int blk = lane + G * j;
                T q[4];
                uint32_t w[2];
                philox_normal4<T>(rng.seed, (uint32_t)blk, gc, gd, q, w);
                if (raw2 && blk == ub) { raw2[0] = w[0]; raw2[1] = w[1]; }
                if (4 * G * (j + 1) <= D) {   // warp-uniform: block j of EVERY lane is real -> no per-element masks
#pragma unroll
                    for (int i = 0; i < 4; ++i) z[4 * j + i] = q[i];
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) z[4 * j + i] = (4 * blk + i < D) ? q[i] : T(0);
                }
            }
        }
    }
    __device__ __forceinline__ T uniform(const bk_rng& rng, int64_t C, int64_t chain, int64_t t,
                                         int k) const {
        if (rng.mode == BK_RNG_INJECTED)
            return reinterpret_cast<const T*>(rng.uniforms)[(t * C + chain) * rng.n_uniform + k];
        return philox_uniform<T>(rng.seed, (uint32_t)k, (uint32_t)(rng.chain_offset + (uint64_t)chain),
                                 (uint32_t)(rng.draw_offset + (uint64_t)t));
    }
};

// Per-lane view of a diagonal Gaussian (MK_ISO keeps nothing per element).
template <typename T, int G, int J, int MK>
struct SepGauss {
    using A = Ar<T>;
    static constexpr int NE = 4 * J;
    T pr[MK == MK_DIAG ? NE : 1];
    T mu[MK == MK_DIAG ? NE : 1];
    T me[MK == MK_DIAG ? NE : 1];
    T prec_scalar;

    __device__ __forceinline__ void init(const SepModel<T>& m, const Lanes<T, G, J>& ln) {
        prec_scalar = m.prec_scalar;
        if constexpr (MK == MK_DIAG) {
            if (m.prec) ln.load(m.prec, pr, T(0));
            else {
#pragma unroll
                for (int k = 0; k < NE; ++k) pr[k] = ln.valid(k) ? m.prec_scalar : T(0);
            }
            if (m.mu) ln.load(m.mu, mu, T(0));
            else {
#pragma unroll
                for (int k = 0; k < NE; ++k) mu[k] = T(0);
            }
            if (m.metric) ln.load(m.metric, me, T(0));
            else {
#pragma unroll
                for (int k = 0; k < NE; ++k) me[k] = T(1);
            }
        }
    }
    // gradient of log p at x (element k)
    __device__ __forceinline__ T grad(const T (&x)[NE], int k) const {
        if constexpr (MK == MK_ISO) return -A::mul(prec_scalar, x[k]);
        else return -A::mul(pr[k], A::sub(x[k], mu[k]));
    }
    // metric * gradient
    __device__ __forceinline__ T mgrad(const T (&x)[NE], int k) const {
        if constexpr (MK == MK_ISO) return grad(x, k);
        else return A::mul(me[k], grad(x, k));
    }
    // log density (group-reduced; identical in every lane of the group)
    __device__ __forceinline__ T logp(const T (&x)[NE]) const {
        T s = T(0);
        if constexpr (MK == MK_ISO) {
#pragma unroll
            for (int k = 0; k < NE; ++k) s = A::add(s, A::mul(x[k], x[k]));
            s = group_sum<G>(s);
            return A::mul(T(-0.5), A::mul(prec_scalar, s));
        } else {
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                T d = A::sub(x[k], mu[k]);
                s = A::add(s, A::mul(d, A::mul(pr[k], d)));
            }
            s = group_sum<G>(s);
            return A::mul(T(-0.5), s);
        }
    }
    // 0.5 * rho . (metric * rho)
    __device__ __forceinline__ T kinetic(const T (&r)[NE]) const {
        T s = T(0);
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            if constexpr (MK == MK_ISO) s = A::add(s, A::mul(r[k], r[k]));
            else s = A::add(s, A::mul(r[k], A::mul(me[k], r[k])));
        }
        s = group_sum<G>(s);
        return A::mul(T(0.5), s);
    }
};

}  // namespace bk
