// DrGhmcDiag (drghmc.py:37-446) as one fused kernel for separable model plugins.
//
// Every chain (a group of G lanes, state in registers) follows its own
// data-dependent schedule: up to K proposals with probabilistic retry, and for
// proposal k the recursive ghost-proposal Hastings terms (worst case 2^k
// leapfrog trajectories, drghmc.py:424-436).  The Python recursion becomes
// compile-time recursion on the proposal index (Accept<k> calls Accept<i<k>),
// so no dynamic stack is needed and shuffles use the group's own lane mask
// (groups of one warp diverge freely).
//
// The reference's (logp, grad) cache stack (drghmc.py:82,243-247) only avoids
// recomputation: a deterministic plugin returns identical values, so the
// kernel recomputes log p and its gradient from the position.
#include <stdlib.h>
#include "drghmc_generic.h"
#include "model.h"
#include "sep_common.cuh"

namespace bk {

constexpr int DR_KMAX = 6;

template <typename T>
struct DrArgs {
    T* theta;
    T* rho;
    int64_t C;
    int D, vec;
    SepModel<T> model;
    int K;
    T eps[DR_KMAX], half_eps[DR_KMAX];
    int cnt[DR_KMAX];
    T s_keep, s_new;  // sqrt(1-damping), sqrt(damping)
    int prob_retry;
    int64_t n_draws;
    bk_rng rng;
    T* draws;
    T* logp;
    int32_t* accept;
    int32_t* n_used;
};

template <int G, typename T>
__device__ __forceinline__ T masked_group_sum(T v, unsigned mask) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;
}

template <typename T, int G, int J, int MK>
struct DrCtx {
    using A = Ar<T>;
    static constexpr int NE = 4 * J;
    const DrArgs<T>& a;
    SepGauss<T, G, J, MK>& md;
    unsigned mask;

    __device__ __forceinline__ T logp(const T (&x)[NE]) const {
        T s = T(0);
        if constexpr (MK == MK_ISO) {
#pragma unroll
            for (int k = 0; k < NE; ++k) s = A::add(s, A::mul(x[k], x[k]));
            s = masked_group_sum<G>(s, mask);
            return A::mul(T(-0.5), A::mul(md.prec_scalar, s));
        } else {
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                T d = A::sub(x[k], md.mu[k]);
                s = A::add(s, A::mul(d, A::mul(md.pr[k], d)));
            }
            s = masked_group_sum<G>(s, mask);
            return A::mul(T(-0.5), s);
        }
    }
    __device__ __forceinline__ T kinetic(const T (&r)[NE]) const {
        T s = T(0);
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            if constexpr (MK == MK_ISO) s = A::add(s, A::mul(r[k], r[k]));
            else s = A::add(s, A::mul(r[k], A::mul(md.me[k], r[k])));
        }
        return A::mul(T(0.5), masked_group_sum<G>(s, mask));
    }
    // drghmc.py:317: bool * float (False * -inf = nan on purpose)
    __device__ __forceinline__ T retry(T reject_logp) const {
        return a.prob_retry ? reject_logp : A::mul(T(0), reject_logp);
    }
    // leapfrog (drghmc.py:253-289) + flip (drghmc.py:345) with proposal-i parameters
    __device__ __forceinline__ void propose(int i, const T (&q0)[NE], const T (&r0)[NE], T (&q)[NE],
                                            T (&r)[NE]) const {
        const T eps = a.eps[i], half = a.half_eps[i];
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            r[k] = A::add(r0[k], A::mul(half, md.mgrad(q0, k)));
            q[k] = A::add(q0[k], A::mul(eps, r[k]));
        }
        for (int s = 1; s < a.cnt[i]; ++s) {
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                r[k] = A::add(r[k], A::mul(eps, md.mgrad(q, k)));
                q[k] = A::add(q[k], A::mul(eps, r[k]));
            }
        }
#pragma unroll
        for (int k = 0; k < NE; ++k) r[k] = -A::add(r[k], A::mul(half, md.mgrad(q, k)));
    }
};

template <typename T>
__device__ __forceinline__ T log1m_exp(T a) {  // np.log1p(-np.exp(a))
    return Ar<T>::log1p_(-Ar<T>::exp_(a));
}

// log acceptance probability of proposal K made from a state with
// (cur_hastings, cur_logp) to (qp, rp)  -- drghmc.py:391-446
template <typename T, int G, int J, int MK, int K>
struct Accept {
    static constexpr int NE = 4 * J;
    using Ctx = DrCtx<T, G, J, MK>;
    using A = Ar<T>;

    template <int I>
    static __device__ __forceinline__ bool ghosts(const Ctx& c, const T (&qp)[NE], const T (&rp)[NE],
                                                  T prop_logp, T& prop_hastings) {
        if constexpr (I < K) {
            T qg[NE], rg[NE];
            c.propose(I, qp, rp, qg, rg);
            T ai, unused;
            Accept<T, G, J, MK, I>::run(c, qg, rg, prop_hastings, prop_logp, ai, unused);
            if (ai == T(0)) return true;  // early exit (drghmc.py:430-432)
            prop_hastings = A::add(prop_hastings, log1m_exp(ai));
            return ghosts<I + 1>(c, qp, rp, prop_logp, prop_hastings);
        } else {
            return false;
        }
    }

    static __device__ __noinline__ void run(const Ctx& c, const T (&qp)[NE], const T (&rp)[NE],
                                            T cur_hastings, T cur_logp, T& a_out, T& prop_logp_out) {
        const T prop_logp = A::sub(c.logp(qp), c.kinetic(rp));
        prop_logp_out = prop_logp;
        T prop_hastings = T(0);
        if (ghosts<0>(c, qp, rp, prop_logp, prop_hastings)) {
            a_out = neg_inf<T>();
            return;
        }
        const T frac = A::add(A::add(A::sub(prop_logp, cur_logp), A::sub(prop_hastings, cur_hastings)),
                              A::sub(c.retry(prop_hastings), c.retry(cur_hastings)));
        a_out = frac < T(0) ? frac : T(0);  // python min(0, frac): nan -> 0
    }
};

template <typename T, int G, int J, int MK, int K>
__device__ __forceinline__ void accept_dispatch(int k, const DrCtx<T, G, J, MK>& c, const T (&qp)[4 * J],
                                                const T (&rp)[4 * J], T ch, T cl, T& a, T& pl) {
    if constexpr (K < DR_KMAX) {
        if (k == K) Accept<T, G, J, MK, K>::run(c, qp, rp, ch, cl, a, pl);
        else accept_dispatch<T, G, J, MK, K + 1>(k, c, qp, rp, ch, cl, a, pl);
    }
}

template <typename T, int G, int J, int MK>
__global__ void __launch_bounds__(128) k_drghmc(DrArgs<T> a) {
    using A = Ar<T>;
    constexpr int NE = 4 * J;
    const int64_t raw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const bool active = raw < a.C;
    const int64_t chain = active ? raw : a.C - 1;
    Lanes<T, G, J> ln;
    ln.lane = threadIdx.x % G;
    ln.D = a.D;
    ln.vec = a.vec != 0;
    SepGauss<T, G, J, MK> md;
    md.init(a.model, ln);
    const int lane32 = threadIdx.x & 31;
    const unsigned mask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane32 / G * G));
    DrCtx<T, G, J, MK> ctx{a, md, mask};

    T th[NE], rho[NE];
    ln.load(a.theta + chain * (int64_t)a.D, th, T(0));
    ln.load(a.rho + chain * (int64_t)a.D, rho, T(0));

    for (int64_t t = 0; t < a.n_draws; ++t) {
        T z[NE];
        ln.normals(a.rng, a.C, chain, t, z);
#pragma unroll
        for (int k = 0; k < NE; ++k)  // drghmc.py:360-364
            rho[k] = A::add(A::mul(rho[k], a.s_keep), A::mul(a.s_new, z[k]));
        T cur_logp = A::sub(ctx.logp(th), ctx.kinetic(rho));
        T cur_hastings = T(0), reject_logp = T(0);
        int ui = 0;
        bool moved = false;
        for (int k = 0; k < a.K; ++k) {
            const T u_retry = ln.uniform(a.rng, a.C, chain, t, ui++);
            if (!(log_u(u_retry) < ctx.retry(reject_logp))) break;  // drghmc.py:369-371
            T qp[NE], rp[NE];
            ctx.propose(k, th, rho, qp, rp);
            T acc_lp, prop_logp;
            accept_dispatch<T, G, J, MK, 0>(k, ctx, qp, rp, cur_hastings, cur_logp, acc_lp, prop_logp);
            const T u_acc = ln.uniform(a.rng, a.C, chain, t, ui++);
            if (log_u(u_acc) < acc_lp) {  // drghmc.py:378-381
#pragma unroll
                for (int e = 0; e < NE; ++e) { th[e] = qp[e]; rho[e] = rp[e]; }
                cur_logp = prop_logp;
                moved = true;
                break;
            }
            reject_logp = log1m_exp(acc_lp);
            cur_hastings = A::add(cur_hastings, reject_logp);
        }
#pragma unroll
        for (int e = 0; e < NE; ++e) rho[e] = -rho[e];  // drghmc.py:388
        if (active) {
            if (a.draws) ln.store(a.draws + (t * a.C + chain) * (int64_t)a.D, th);
            if (ln.lane == 0) {
                if (a.logp) a.logp[t * a.C + chain] = cur_logp;
                if (a.accept) a.accept[t * a.C + chain] = moved ? 1 : 0;
                if (a.n_used) a.n_used[t * a.C + chain] = ui;
            }
        }
    }
    if (active) {
        ln.store(a.theta + chain * (int64_t)a.D, th);
        ln.store(a.rho + chain * (int64_t)a.D, rho);
    }
}

template <typename T, int G, int J, int MK>
static int launch_dr(const DrArgs<T>& a, cudaStream_t st) {
    const int64_t per_block = 128 / G;
    const int64_t blocks = (a.C + per_block - 1) / per_block;
    k_drghmc<T, G, J, MK><<<(unsigned)blocks, 128, 0, st>>>(a);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

template <typename T, int MK>
static int launch_dr_mk(const DrArgs<T>& a, cudaStream_t st) {
    const int D = a.D;
    if (D <= 4) return launch_dr<T, 1, 1, MK>(a, st);
    if (D <= 16) return launch_dr<T, 4, 1, MK>(a, st);
    if (D <= 32) return launch_dr<T, 8, 1, MK>(a, st);
    // fp32: 8 lanes x 16 elements per chain (see sampler_sep.cu: same Philox blocks, a quarter of the per-lane overhead)
    static int wide = -1;
    if (wide < 0) { const char* e = getenv("BK_SEP_WIDE"); wide = (e && e[0] == '0') ? 0 : 1; }
    if (sizeof(T) == 4 && wide && D > 64 && D <= 128) return launch_dr<T, 8, 4, MK>(a, st);
    if (sizeof(T) == 4 && wide && D > 32 && D <= 64) return launch_dr<T, 4, 4, MK>(a, st);
    if (D <= 64) return launch_dr<T, 16, 1, MK>(a, st);
    if (D <= 128) return launch_dr<T, 32, 1, MK>(a, st);
    if (D <= 256) return launch_dr<T, 32, 2, MK>(a, st);
    set_error("bk_drghmc_sample supports D <= 256 (got %d)", D);
    return BK_E_UNSUPPORTED;
}

template <typename T>
static int drghmc_t(const Model& m, void* theta, void* rho, int64_t C, int K, const double* sizes,
                    const int32_t* counts, double damping, int prob_retry, const void* metric,
                    int64_t n, const bk_rng* rng, const bk_draw_out& out, int32_t* n_used,
                    cudaStream_t st) {
    DrArgs<T> a;
    memset(&a, 0, sizeof(a));
    a.theta = (T*)theta;
    a.rho = (T*)rho;
    a.C = C;
    a.D = (int)m.d.dims;
    a.model.mu = (const T*)m.d.mu;
    a.model.prec = (const T*)m.d.prec;
    a.model.prec_scalar = (T)(1.0 / (m.d.sigma * m.d.sigma));
    a.model.metric = (const T*)metric;
    a.K = K;
    for (int k = 0; k < K; ++k) {
        a.eps[k] = (T)sizes[k];
        a.half_eps[k] = (T)(0.5 * sizes[k]);
        a.cnt[k] = counts[k];
    }
    a.s_keep = (T)sqrt(1 - damping);
    a.s_new = (T)sqrt(damping);
    a.prob_retry = prob_retry;
    a.n_draws = n;
    a.rng = *rng;
    a.draws = (T*)out.draws;
    a.logp = (T*)out.logp;
    a.accept = out.accept;
    a.n_used = n_used;
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    a.vec = (a.D % 4 == 0 && al(theta) && al(rho) && al(out.draws) && al(m.d.mu) && al(m.d.prec) &&
             al(metric) && (rng->mode != BK_RNG_INJECTED || al(rng->normals))) ? 1 : 0;
    const bool iso = !a.model.mu && !a.model.prec && !a.model.metric;
    return iso ? launch_dr_mk<T, MK_ISO>(a, st) : launch_dr_mk<T, MK_DIAG>(a, st);
}

}  // namespace bk

using namespace bk;

extern "C" {

// the fused register-resident kernel serves iso / diagonal Gaussian plugins up to 256 dims, the runtime-compiled
// bk_user_drghmc (user_model.cu) user models up to USER_FUSED_MAX_D; everything else (dense precision, logistic
// regression, binomial, D > 256, larger user models) runs on the lockstep engine of drghmc_generic.cu
static bool drghmc_fused(const Model& m) { return !force_generic() && m.separable() && m.d.dims <= 256; }
static bool drghmc_user_fused(const Model& m) { return !force_generic() && user_fused(m); }

size_t bk_drghmc_workspace_bytes(uint64_t handle, int64_t C, int32_t max_proposals) {
    const Model* m = get_model(handle);
    if (!m || drghmc_fused(*m) || drghmc_user_fused(*m)) return 0;
    return drghmc_generic_ws_bytes(*m, C, max_proposals);
}

int bk_drghmc_cuda_prepare(uint64_t handle, char* log_out, size_t log_bytes) {
    if (log_out && log_bytes) log_out[0] = '\0';
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    return drghmc_user_fused(*m) ? user_drghmc_prepare(*m, log_out, log_bytes) : BK_OK;
}

int bk_drghmc_sample(uint64_t handle, void* theta, void* rho, int64_t C, int32_t max_proposals,
                     const double* step_sizes_host, const int32_t* step_counts_host, double damping,
                     int32_t prob_retry, const void* metric, int64_t n_draws, const bk_rng* rng,
                     const bk_draw_out* out, int32_t* n_uniform_used_out, void* ws, size_t ws_bytes,
                     void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && rho && C >= 0 && n_draws >= 0, "bk_drghmc_sample: bad theta/rho/C/n_draws");
    BK_CHECK_ARG(max_proposals >= 1, "max_proposals must be greater than or equal to 1, not %d",
                 max_proposals);
    BK_CHECK_ARG(step_sizes_host && step_counts_host, "bk_drghmc_sample: step sizes/counts required");
    for (int k = 0; k < max_proposals; ++k) {
        BK_CHECK_ARG(step_sizes_host[k] > 0, "each step size in leapfrog_step_sizes must be positive, "
                     "but found step size of %g at index %d", step_sizes_host[k], k);
        BK_CHECK_ARG(step_counts_host[k] > 0, "each step count in leapfrog_step_counts must be "
                     "positive, but found step count of %d at index %d", step_counts_host[k], k);
    }
    BK_CHECK_ARG(damping > 0 && damping <= 1, "damping must be within (0, 1], but found damping of %g",
                 damping);
    BK_CHECK_ARG(rng && (rng->mode == BK_RNG_PHILOX ||
                         (rng->normals && rng->uniforms && rng->n_uniform >= 2 * max_proposals)),
                 "bk_drghmc_sample: injected rng needs normals, uniforms and n_uniform >= 2K");
    if (max_proposals > DR_KMAX) {
        set_error("bk_drghmc_sample supports max_proposals <= %d (got %d)", DR_KMAX, max_proposals);
        return BK_E_UNSUPPORTED;
    }
    bk_draw_out o = out ? *out : bk_draw_out{nullptr, nullptr, nullptr};
    if (C == 0 || n_draws == 0) return BK_OK;
    if (drghmc_user_fused(*m))
        return user_drghmc_sample(*m, theta, rho, C, max_proposals, step_sizes_host, step_counts_host, damping,
                                  prob_retry, metric, n_draws, rng, o, n_uniform_used_out, (cudaStream_t)stream);
    if (!drghmc_fused(*m))
        return drghmc_generic(*m, theta, rho, C, max_proposals, step_sizes_host, step_counts_host, damping, prob_retry,
                              metric, n_draws, rng, o, n_uniform_used_out, ws, ws_bytes, (cudaStream_t)stream);
    if (m->d.dtype == BK_F64)
        return drghmc_t<double>(*m, theta, rho, C, max_proposals, step_sizes_host, step_counts_host,
                                damping, prob_retry, metric, n_draws, rng, o, n_uniform_used_out,
                                (cudaStream_t)stream);
    return drghmc_t<float>(*m, theta, rho, C, max_proposals, step_sizes_host, step_counts_host, damping,
                           prob_retry, metric, n_draws, rng, o, n_uniform_used_out, (cudaStream_t)stream);
}

}  // extern "C"
