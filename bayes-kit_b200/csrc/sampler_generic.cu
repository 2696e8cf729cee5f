// Generic (model-agnostic) sampler engine: HMCDiag / MALA / random-walk
// Metropolis as short sequences of row kernels around a batched device
// gradient evaluation (model_eval).  Serves every model plugin in fp64 parity
// mode and is the fp32 fallback for models without a fused kernel.
//
// Reference semantics: hmc.py:36-63, mala.py:40-79, metropolis.py:12-135.
// State cached between draws: (lp, grad) at theta -- the reference recomputes
// them (hmc.py:57,45) but a deterministic model returns identical values.
#include "sampler_generic.h"

namespace bk {

// One warp per chain; lane b-strided blocks of 4 elements (matches the Philox
// element-block mapping of the fused kernels, so results do not depend on the
// engine that ran).
template <typename T>
struct Row {
    const bk_rng& rng;
    int64_t C, c, t;
    int D, lane;
    __device__ __forceinline__ void normal4(int b, T (&z)[4]) const {
        if (rng.mode == BK_RNG_INJECTED) {
            const T* p = reinterpret_cast<const T*>(rng.normals) + (t * C + c) * (int64_t)D;
#pragma unroll
            for (int i = 0; i < 4; ++i) z[i] = (4 * b + i < D) ? p[4 * b + i] : T(0);
        } else {
            philox_normal4<T>(rng.seed, (uint32_t)b, (uint32_t)(rng.chain_offset + (uint64_t)c),
                              (uint32_t)(rng.draw_offset + (uint64_t)t), z);
        }
    }
    __device__ __forceinline__ T uniform(int k) const {
        if (rng.mode == BK_RNG_INJECTED)
            return reinterpret_cast<const T*>(rng.uniforms)[(t * C + c) * rng.n_uniform + k];
        if (k == 0 && rng.n_uniform == 1)      // the samplers' accept uniform: one rule for every engine
            return philox_accept_uniform<T>(rng.seed, (uint32_t)(rng.chain_offset + (uint64_t)c),
                                            (uint32_t)(rng.draw_offset + (uint64_t)t), D);
        return philox_uniform<T>(rng.seed, (uint32_t)k, (uint32_t)(rng.chain_offset + (uint64_t)c),
                                 (uint32_t)(rng.draw_offset + (uint64_t)t));
    }
};

#define ROW_PROLOGUE()                                                              \
    using A = Ar<T>;                                                                \
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;       \
    const int lane = threadIdx.x & 31;                                              \
    if (c >= p.C) return;                                                           \
    const int D = p.D;                                                              \
    const int64_t off = c * (int64_t)D;                                             \
    (void)lane; (void)off;

// ---- HMC ----------------------------------------------------------------------
// begin: rho ~ N(0,I); H0 = lp - 0.5 rho.(m rho); r = rho - (eps/2) m g
//        [+ first kick/drift if L > 0: r += eps m g ; q = theta + eps r]
template <typename T>
__global__ void k_hmc_begin(GenArgs<T> p, int64_t t) {
    ROW_PROLOGUE();
    Row<T> row{p.rng, p.C, c, t, D, lane};
    T kin = T(0);
    for (int b = lane; 4 * b < D; b += 32) {
        T z[4];
        row.normal4(b, z);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int e = 4 * b + i;
            if (e >= D) break;
            T m = p.metric ? p.metric[e] : T(1);
            T mg = p.metric ? A::mul(m, p.grad[off + e]) : p.grad[off + e];
            kin = A::add(kin, A::mul(z[i], p.metric ? A::mul(m, z[i]) : z[i]));
            T r = A::sub(z[i], A::mul(p.half_eps, mg));
            T q = p.theta[off + e];
            if (p.L > 0) {
                r = A::add(r, A::mul(p.eps, mg));
                q = A::add(q, A::mul(p.eps, r));
            }
            p.r[off + e] = r;
            p.q[off + e] = q;
        }
    }
    kin = warp_sum(kin);
    if (lane == 0) p.h0[c] = A::sub(p.lp[c], A::mul(T(0.5), kin));
}

// step: r += eps m g(q) ; q += eps r     (g(q) in grad_q)
template <typename T>
__global__ void k_hmc_step(GenArgs<T> p) {
    ROW_PROLOGUE();
    for (int e = lane; e < D; e += 32) {
        T g = p.grad_q[off + e];
        T mg = p.metric ? A::mul(p.metric[e], g) : g;
        T r = A::add(p.r[off + e], A::mul(p.eps, mg));
        p.r[off + e] = r;
        p.q[off + e] = A::add(p.q[off + e], A::mul(p.eps, r));
    }
}

// end: r += (eps/2) m g(q); H1; Metropolis test; commit
template <typename T>
__global__ void k_hmc_end(GenArgs<T> p, int64_t t) {
    ROW_PROLOGUE();
    Row<T> row{p.rng, p.C, c, t, D, lane};
    const T* gq = p.L > 0 ? p.grad_q : p.grad;
    const T lpq = p.L > 0 ? p.lp_q[c] : p.lp[c];
    T kin = T(0);
    for (int e = lane; e < D; e += 32) {
        T g = gq[off + e];
        T m = p.metric ? p.metric[e] : T(1);
        T mg = p.metric ? A::mul(m, g) : g;
        T r = A::add(p.r[off + e], A::mul(p.half_eps, mg));
        kin = A::add(kin, A::mul(r, p.metric ? A::mul(m, r) : r));
    }
    kin = warp_sum(kin);
    const T h1 = A::sub(lpq, A::mul(T(0.5), kin));
    const T h0 = p.h0[c];
    const bool acc = log_u(row.uniform(0)) < A::sub(h1, h0);
    T* dr = p.draws ? p.draws + (t * p.C + c) * (int64_t)D : nullptr;
    for (int e = lane; e < D; e += 32) {
        T v;
        if (acc) {
            v = p.q[off + e];
            p.theta[off + e] = v;
            if (p.L > 0) p.grad[off + e] = gq[off + e];
        } else {
            v = p.theta[off + e];
        }
        if (dr) dr[e] = v;
    }
    if (lane == 0) {
        if (acc && p.L > 0) p.lp[c] = lpq;
        if (p.logp) p.logp[t * p.C + c] = acc ? h1 : h0;
        if (p.accept) p.accept[t * p.C + c] = acc ? 1 : 0;
    }
}

// ---- MALA -----------------------------------------------------------------------
template <typename T>
__global__ void k_mala_propose(GenArgs<T> p, int64_t t) {
    ROW_PROLOGUE();
    Row<T> row{p.rng, p.C, c, t, D, lane};
    for (int b = lane; 4 * b < D; b += 32) {
        T z[4];
        row.normal4(b, z);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int e = 4 * b + i;
            if (e >= D) break;
            p.q[off + e] = A::add(A::add(p.theta[off + e], A::mul(p.eps, p.grad[off + e])),
                                  A::mul(p.sd, z[i]));
        }
    }
}

template <typename T>
__global__ void k_mala_accept(GenArgs<T> p, int64_t t) {
    ROW_PROLOGUE();
    Row<T> row{p.rng, p.C, c, t, D, lane};
    T sf = T(0), sr = T(0);
    for (int e = lane; e < D; e += 32) {
        T th = p.theta[off + e], q = p.q[off + e];
        T df = A::sub(A::sub(q, th), A::mul(p.eps, p.grad[off + e]));
        T dr = A::sub(A::sub(th, q), A::mul(p.eps, p.grad_q[off + e]));
        sf = A::add(sf, A::mul(df, df));
        sr = A::add(sr, A::mul(dr, dr));
    }
    const T fwd = A::mul(p.coef, warp_sum(sf)), rev = A::mul(p.coef, warp_sum(sr));
    const T lp = p.lp[c], lpq = p.lp_q[c];
    const bool acc = log_u(row.uniform(0)) < A::add(A::sub(lpq, lp), A::sub(rev, fwd));
    T* dr = p.draws ? p.draws + (t * p.C + c) * (int64_t)D : nullptr;
    for (int e = lane; e < D; e += 32) {
        T v;
        if (acc) {
            v = p.q[off + e];
            p.theta[off + e] = v;
            p.grad[off + e] = p.grad_q[off + e];
        } else {
            v = p.theta[off + e];
        }
        if (dr) dr[e] = v;
    }
    if (lane == 0) {
        if (acc) p.lp[c] = lpq;
        if (p.logp) p.logp[t * p.C + c] = acc ? lpq : lp;
        if (p.accept) p.accept[t * p.C + c] = acc ? 1 : 0;
    }
}

// ---- random-walk Metropolis(-Hastings) --------------------------------------------
template <typename T>
__global__ void k_mh_propose(GenArgs<T> p, int64_t t) {
    ROW_PROLOGUE();
    Row<T> row{p.rng, p.C, c, t, D, lane};
    for (int b = lane; 4 * b < D; b += 32) {
        T z[4];
        row.normal4(b, z);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int e = 4 * b + i;
            if (e >= D) break;
            p.q[off + e] = A::add(p.theta[off + e], A::mul(p.scale, z[i]));
        }
    }
}

// GRAD (gradient proposals): an accepted chain also takes grad log p(q) into the gradient cache
template <typename T, bool GRAD = false>
__global__ void k_mh_accept(GenArgs<T> p, int64_t t) {
    ROW_PROLOGUE();
    Row<T> row{p.rng, p.C, c, t, D, lane};
    const T lp = p.lp[c], lpq = p.lp_q[c];
    T ratio = A::sub(lpq, lp);
    if (p.dh) {
        ratio = A::add(ratio, p.dh[c]);
    } else if (p.hastings) {
        T sf = T(0), sr = T(0);
        for (int e = lane; e < D; e += 32) {
            T df = A::sub(p.q[off + e], p.theta[off + e]), dr = A::sub(p.theta[off + e], p.q[off + e]);
            sf = A::add(sf, A::mul(df, df));
            sr = A::add(sr, A::mul(dr, dr));
        }
        const T fwd = A::mul(T(-0.5), warp_sum(sf)) / p.s2, rev = A::mul(T(-0.5), warp_sum(sr)) / p.s2;
        ratio = A::add(ratio, A::sub(rev, fwd));
    }
    const bool acc = log_u(row.uniform(0)) < ratio;
    T* dr = p.draws ? p.draws + (t * p.C + c) * (int64_t)D : nullptr;
    for (int e = lane; e < D; e += 32) {
        T v;
        if (acc) {
            v = p.q[off + e];
            p.theta[off + e] = v;
            if constexpr (GRAD) p.grad[off + e] = p.grad_q[off + e];
        } else {
            v = p.theta[off + e];
        }
        if (dr) dr[e] = v;
    }
    if (lane == 0) {
        if (acc) p.lp[c] = lpq;
        if (p.logp) p.logp[t * p.C + c] = acc ? lpq : lp;
        if (p.accept) p.accept[t * p.C + c] = acc ? 1 : 0;
    }
}

// ---- host loops ------------------------------------------------------------------
template <typename T>
size_t generic_ws_bytes(const Model& m, int64_t C) {
    size_t n = (size_t)C * m.d.dims;
    // q, r, grad_q [C,D]; lp_q, h0 [C]; model eval scratch
    return 3 * align_up(n * sizeof(T), 256) + 2 * align_up((size_t)C * sizeof(T), 256) +
           model_eval_ws_bytes(m, C) + 1024;
}
template size_t generic_ws_bytes<float>(const Model&, int64_t);
template size_t generic_ws_bytes<double>(const Model&, int64_t);

template <typename T>
static int carve(const Model& m, GenArgs<T>& p, void* ws, size_t ws_bytes, void** eval_ws,
                 size_t* eval_bytes) {
    Arena ar(ws, ws_bytes);
    size_t n = (size_t)p.C * p.D;
    p.q = ar.take<T>(n);
    p.r = ar.take<T>(n);
    p.grad_q = ar.take<T>(n);
    p.lp_q = ar.take<T>(p.C);
    p.h0 = ar.take<T>(p.C);
    *eval_bytes = model_eval_ws_bytes(m, p.C);
    *eval_ws = ar.take<char>(*eval_bytes);
    if (!ar.ok()) {
        set_error("sampler workspace too small: need %zu bytes, got %zu", ar.off, ws_bytes);
        return BK_E_WORKSPACE;
    }
    return BK_OK;
}

template <typename T>
int run_generic(const Model& m, GenArgs<T> p, int algo, int* cache_valid, void* ws, size_t ws_bytes,
                cudaStream_t st, const MhProposeHook* propose) {
    if (p.C == 0 || p.n_draws == 0) return BK_OK;
    void* ews;
    size_t ebytes;
    int rc = carve(m, p, ws, ws_bytes, &ews, &ebytes);
    if (rc) return rc;
    const unsigned blocks = (unsigned)((p.C * 32 + 255) / 256);
    const bool gradient = propose && propose->gradient;   // a gradient proposal: ALGO_MHRW keeps grad too
    const bool need_grad = algo != ALGO_MHRW || gradient;
    const bool fast = algo == ALGO_HMC && model_has_fast_path(m);
    if (!cache_valid || !*cache_valid) {
        if (fast) {   // same convention as inside the loop: tensor-core gradient, precise density
            rc = model_eval(m, p.theta, p.C, nullptr, p.grad, ews, ebytes, st, false);
            if (rc) return rc;
            rc = model_eval(m, p.theta, p.C, p.lp, nullptr, ews, ebytes, st, true);
        } else {
            rc = model_eval(m, p.theta, p.C, p.lp, need_grad ? p.grad : nullptr, ews, ebytes, st);
        }
        if (rc) return rc;
        if (cache_valid) *cache_valid = 1;
    }
    for (int64_t t = 0; t < p.n_draws; ++t) {
        if (algo == ALGO_HMC) {
            k_hmc_begin<T><<<blocks, 256, 0, st>>>(p, t);
            BK_LAUNCH_CHECK();
            int s_first = 0;
            if constexpr (sizeof(T) == 4) {
                // regression plugin, interior steps: tensor-core gradient + finish + kick + drift + next bf16
                // operand, all L - 1 of them in one persistent launch -- logreg_tc.cu
                if (fast && m.d.kind == BK_MODEL_HIER_LOGREG && p.L > 1) {
                    rc = hlr_tc_interior_steps(m, (float*)p.q, (float*)p.r, p.C, (float)p.eps,
                                               (const float*)p.metric, p.L - 1, ews, ebytes, st);
                    if (rc) return rc;
                    s_first = p.L - 1;
                }
            }
            for (int s = s_first; s < p.L; ++s) {
                // Gradients may come from the plugin's reduced-precision tensor-core path at
                // EVERY step: leapfrog with any deterministic gradient function is reversible
                // and volume preserving (the endpoint gradient is also what the next
                // trajectory starts from).  Only the log density that enters the Hamiltonian
                // must be precise: at the endpoint it is evaluated separately, density only.
                if (fast) {
                    rc = model_eval(m, p.q, p.C, nullptr, p.grad_q, ews, ebytes, st, /*precise=*/false);
                    if (rc) return rc;
                    if (s + 1 == p.L) rc = model_eval(m, p.q, p.C, p.lp_q, nullptr, ews, ebytes, st, true);
                } else {
                    rc = model_eval(m, p.q, p.C, p.lp_q, p.grad_q, ews, ebytes, st, true);
                }
                if (rc) return rc;
                if (s + 1 < p.L) {
                    k_hmc_step<T><<<blocks, 256, 0, st>>>(p);
                    BK_LAUNCH_CHECK();
                }
            }
            k_hmc_end<T><<<blocks, 256, 0, st>>>(p, t);
            BK_LAUNCH_CHECK();
        } else if (algo == ALGO_MALA) {
            k_mala_propose<T><<<blocks, 256, 0, st>>>(p, t);
            BK_LAUNCH_CHECK();
            rc = model_eval(m, p.q, p.C, p.lp_q, p.grad_q, ews, ebytes, st);
            if (rc) return rc;
            k_mala_accept<T><<<blocks, 256, 0, st>>>(p, t);
            BK_LAUNCH_CHECK();
        } else {
            if (propose) {
                rc = propose->fn(propose->ctx, p.theta, p.grad, p.q, p.dh, t, st);
                if (rc) return rc;
            } else {
                k_mh_propose<T><<<blocks, 256, 0, st>>>(p, t);
                BK_LAUNCH_CHECK();
            }
            rc = model_eval(m, p.q, p.C, p.lp_q, gradient ? p.grad_q : nullptr, ews, ebytes, st);
            if (rc) return rc;
            if (gradient) {
                if (p.dh) {
                    rc = propose->hastings(propose->ctx, p.theta, p.q, p.grad_q, p.dh, st);
                    if (rc) return rc;
                }
                k_mh_accept<T, true><<<blocks, 256, 0, st>>>(p, t);
            } else {
                k_mh_accept<T><<<blocks, 256, 0, st>>>(p, t);
            }
            BK_LAUNCH_CHECK();
        }
    }
    return BK_OK;
}

template int run_generic<float>(const Model&, GenArgs<float>, int, int*, void*, size_t, cudaStream_t,
                                const MhProposeHook*);
template int run_generic<double>(const Model&, GenArgs<double>, int, int*, void*, size_t, cudaStream_t,
                                 const MhProposeHook*);

}  // namespace bk
