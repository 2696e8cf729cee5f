// TemperedLikelihoodSMC hot path (smc.py:12-89):
//   bk_smc_move_weight       -- RW-Metropolis move at time(n-1) fused with the
//                               importance log-weights lp_n - lp_{n-1}
//   bk_smc_weight_stats      -- max / sum exp / sum exp^2 (log-sum-exp normaliser, ESS)
//   bk_smc_resample_indices  -- normalise, block scan -> CDF, binary search
//                               (multinomial = np.random.choice; systematic)
//   bk_gather_rows           -- thetas[idx]
#include <stdlib.h>

#include "model.h"
#include "sep_common.cuh"
#include "smc_shard.cuh"
#include "user_kernels.cuh"

namespace bk {

enum { SMC_MODEL_GPL = 0, SMC_MODEL_BINOM = 1 };

template <typename T>
struct SmcArgs {
    T* thetas;                 // [M, D] moved particles (out)
    const T* src;              // particles to move: row src_idx[m] (the pending resample) or row m
    const int64_t* src_idx;    // [M] or NULL
    int64_t M;
    int D, vec, vec2;
    const T *mu, *pl, *m0, *p0;   // GAUSS_PRIOR_LIK
    T bp[6];                      // BINOMIAL_LOGIT: alpha, beta, x, N, log C(N, x), log B(alpha, beta)
    T t0, t1;
    T scale;                   // RW: proposal sd (smc.py:81); MALA: epsilon (mala.py:41-45); HMC: stepsize
    int steps;                 // HMC: leapfrog steps
    bk_rng rng;
    T* logw;
    const T* logw_prev;        // [M] log-weights carried from temperatures without resampling, or NULL
    int32_t* accept;
    // ---- sharded particle system (smc_shard.cuh); sh.world == 0: plain single-array call ----
    ShardGeom sh;              // src_idx holds GLOBAL particle ids, row gid lives on rank owner(gid)
    const T* src_tab[BK_SMC_MAX_WORLD];   // peer-accessible particle arrays the ids refer to
    uint64_t* mail_tab[BK_SMC_MAX_WORLD]; // every rank's mailbox (mail_tab[sh.rank] = ours)
    uint64_t epoch;            // this temperature step's message number
    uint64_t wait_done;        // > 0: wait until every rank's "indices of step wait_done are final" arrived
    double* maxpart;           // [gridDim.x] per-CTA maxima of the log-weights (NULL: no statistics epilogue)
    unsigned* ticket;
    // (log_likelihood, log_prior) carried with the particle: written for every moved particle (llpr_out [M, 2]);
    // read from the parent's pair (llpr_tab[owner][row]) instead of re-evaluating the model when carry != 0
    T* llpr_out;
    const T* llpr_tab[BK_SMC_MAX_WORLD];
    int carry;
};

// ---- per-lane views of the LogPriorLikelihoodModel plugins (typing.py:37-42) ------------------
// terms(): log_likelihood and log_prior of x (group-reduced); gll / gpr: their elementwise gradients.
// The tempered density of smc.py:47-51 is lp_t = ll * t + prior, its gradient gll * t + gpr.
template <typename T, int G, int J>
struct GplView {
    using A = Ar<T>;
    static constexpr int NE = 4 * J;
    T mu[NE], pl[NE], m0[NE], p0[NE];
    template <typename LN>
    __device__ __forceinline__ void init(const SmcArgs<T>& a, const LN& ln) {
        ln.load(a.mu, mu, T(0));
        ln.load(a.pl, pl, T(0));
        ln.load(a.m0, m0, T(0));
        ln.load(a.p0, p0, T(0));
    }
    __device__ __forceinline__ void terms(const T (&x)[NE], T& ll, T& pr) const {
        T s = T(0), s2 = T(0);
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            T dl = A::sub(x[k], mu[k]), dp = A::sub(x[k], m0[k]);
            s = A::add(s, A::mul(A::mul(pl[k], dl), dl));
            s2 = A::add(s2, A::mul(A::mul(p0[k], dp), dp));
        }
        ll = A::mul(T(-0.5), group_sum<G>(s));
        pr = A::mul(T(-0.5), group_sum<G>(s2));
    }
    __device__ __forceinline__ T gll(const T (&x)[NE], int k) const { return -A::mul(pl[k], A::sub(x[k], mu[k])); }
    __device__ __forceinline__ T gpr(const T (&x)[NE], int k) const { return -A::mul(p0[k], A::sub(x[k], m0[k])); }
};

// Beta-binomial on the logit scale (the reference's own SMC test target, test/models/binomial.py:46-54):
//   p = inv_logit(theta);  ll = log C(N, x) + x log p + (N - x) log(1 - p)
//   prior = Beta(p; alpha, beta) with the Jacobian log p + log(1 - p) = alpha log p + beta log(1 - p) - log B
// D == 1: one lane per particle, only element 0 is live.
template <typename T>
__device__ __forceinline__ void logit_logs(T th, T& lp1, T& l1m, T& p) {
    using A = Ar<T>;
    const T e = A::exp_(-fabs(th));             // exp(-|theta|)
    const T l = A::log1p_(e);
    lp1 = th >= T(0) ? -l : A::sub(th, l);      // log p     = -softplus(-theta)
    l1m = th >= T(0) ? A::sub(-th, l) : -l;     // log (1-p) = -softplus(theta)
    p = th >= T(0) ? T(1) / A::add(T(1), e) : e / A::add(T(1), e);
}
template <typename T, int G, int J>
struct BinomView {
    using A = Ar<T>;
    static constexpr int NE = 4 * J;
    T al, be, xs, Nn, lch, lbe;
    template <typename LN>
    __device__ __forceinline__ void init(const SmcArgs<T>& a, const LN&) {
        al = a.bp[0]; be = a.bp[1]; xs = a.bp[2]; Nn = a.bp[3]; lch = a.bp[4]; lbe = a.bp[5];
    }
    __device__ __forceinline__ void terms(const T (&x)[NE], T& ll, T& pr) const {
        T lp1, l1m, p;
        logit_logs<T>(x[0], lp1, l1m, p);
        ll = A::add(A::add(lch, A::mul(xs, lp1)), A::mul(A::sub(Nn, xs), l1m));
        pr = A::sub(A::add(A::mul(al, lp1), A::mul(be, l1m)), lbe);
    }
    __device__ __forceinline__ T gll(const T (&x)[NE], int k) const {
        if (k != 0) return T(0);
        T lp1, l1m, p;
        logit_logs<T>(x[0], lp1, l1m, p);
        return A::sub(xs, A::mul(Nn, p));
    }
    __device__ __forceinline__ T gpr(const T (&x)[NE], int k) const {
        if (k != 0) return T(0);
        T lp1, l1m, p;
        logit_logs<T>(x[0], lp1, l1m, p);
        return A::sub(al, A::mul(A::add(al, be), p));
    }
};

// Persistent groups: a group of G lanes owns elements 4*lane..4*lane+3 (per j) of EVERY particle it
// visits, so the model's per-dimension parameters are loaded once and stay in registers.  The
// resample index and the particle row of the NEXT visit are requested before the current particle is
// processed (two dependent global loads deep), the accept uniform is drawn by the group's first lane only.
// MOVE selects the Markov kernel applied at temperature t0 = time(n-1) (smc.py:54-57).
// VM: row access mode fixed at compile time (sep_common.cuh) for the hot layout; -1 = run-time flags.  (c4: 20.4 -> 17.8 ms.
// Measured and dropped: the model's per-dimension parameters in shared memory instead of registers -- the same 17.8 ms
// at 3 CTAs / SM, and 22.2 / 26.7 ms at 4 / 5 CTAs per SM, where the register cap spills.)
template <typename T, int G, int J, template <typename, int, int> class View, int MOVE, int OCC = 0, int VM = -1>
__global__ void __launch_bounds__(128, OCC ? OCC : (J >= 4 && sizeof(T) == 4) ? 3 : (J == 2 && G == 8) ? 5 : 1) k_smc_move_weight(SmcArgs<T> a) {
    using A = Ar<T>;
    constexpr int NE = 4 * J;
    const int64_t n_groups = (int64_t)gridDim.x * blockDim.x / G;
    const int64_t g0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int64_t n_it = (a.M + n_groups - 1) / n_groups;       // same trip count for every lane of a warp
    Lanes<T, G, J, VM> ln;
    ln.lane = threadIdx.x % G;
    ln.D = a.D;
    ln.vec = a.vec != 0;
    ln.vec2 = a.vec2 != 0;
    View<T, G, J> md;
    md.init(a, ln);
    const int ub = accept_block(a.D);   // common.cuh: the accept uniform = words of element block ceil(D / 4) of the normal stream
    const bool spare_block = a.rng.mode == BK_RNG_PHILOX && ub < G * J;
    auto particle = [&](int64_t it) { const int64_t r = g0 + it * n_groups; return r < a.M ? r : a.M - 1; };
    auto row_of = [&](int64_t m) { return a.src_idx ? a.src_idx[m] : m; };
    // sharded source: the resample indices are global particle ids; the row is read from its owner's
    // array over NVLink peer memory (no all-gather of particles, no all_to_all)
    const bool sharded = a.sh.world > 1 && a.src_idx != nullptr;
    auto row_ptr = [&](int64_t gid) -> const T* {
        if (!sharded) return a.src + gid * (int64_t)a.D;
        int r; int64_t loc;
        shard_locate(a.sh, gid, r, loc);
        return a.src_tab[r] + loc * (int64_t)a.D;
    };
    auto llpr_ptr = [&](int64_t gid) -> const T* {
        if (!sharded) return a.llpr_tab[a.sh.world > 0 ? a.sh.rank : 0] + 2 * gid;
        int r; int64_t loc;
        shard_locate(a.sh, gid, r, loc);
        return a.llpr_tab[r] + 2 * loc;
    };
    const bool carry = a.carry != 0;
    if (a.wait_done) {   // the indices (and the rows they point at) of the previous step are final on every rank
        if ((int)threadIdx.x < a.sh.world)
            mail_wait(a.mail_tab[a.sh.rank] + MB_DONE + (a.wait_done & 1) * BK_SMC_MAX_WORLD + threadIdx.x, a.wait_done,
                      a.mail_tab[a.sh.rank]);
        __syncthreads();
    }
    T nx[NE];                                  // particle of the next visit
    int64_t row_nn = 0;                        // resample index of the visit after that
    double lw_max = -INFINITY;
    T nll = T(0), npr = T(0);                  // parent's (ll, prior) of the next visit
    if (n_it > 0) {
        const int64_t r0 = row_of(particle(0));
        ln.load(row_ptr(r0), nx, T(0));
        if (carry) { const T* lp2 = llpr_ptr(r0); nll = lp2[0]; npr = lp2[1]; }
    }
    if (n_it > 1) row_nn = row_of(particle(1));
    const T t0 = a.t0;
    auto tgrad = [&](const T (&x)[NE], int k) { return A::add(A::mul(md.gll(x, k), t0), md.gpr(x, k)); };
    for (int64_t it = 0; it < n_it; ++it) {
        const int64_t raw = g0 + it * n_groups;
        const bool active = raw < a.M;
        const int64_t m = active ? raw : a.M - 1;
        T th[NE], z[NE], st[NE];
#pragma unroll
        for (int k = 0; k < NE; ++k) th[k] = nx[k];
        T ll_c = nll, pr_c = npr;
        // thetas[idxs] of the previous importance_resample (smc.py:75) is folded into this read
        if (it + 1 < n_it) {
            ln.load(row_ptr(row_nn), nx, T(0));
            if (carry) { const T* lp2 = llpr_ptr(row_nn); nll = lp2[0]; npr = lp2[1]; }
        }
        if (it + 2 < n_it) row_nn = row_of(particle(it + 2));
        uint32_t raw2[2] = {0u, 0u};
        ln.normals(a.rng, a.M, m, 0, z, raw2, ub);
        // accept uniform: when the lane layout has a slot for block ub, the pass above made its Philox words --
        // one counter-mode call per lane and particle instead of two.  Otherwise one extra call (same block);
        // injected streams: the recorded uniform.
        T lu = T(0);
        if (spare_block) {
            if (ln.lane == ub % G) {
                if constexpr (sizeof(T) == 4) lu = log_u(u01(raw2[0]));
                else lu = log_u(u01d(raw2[0], raw2[1]));
            }
            lu = __shfl_sync(0xffffffffu, lu, ub % G, G);
        } else {
            if (ln.lane == 0)
                lu = log_u(a.rng.mode == BK_RNG_PHILOX
                               ? philox_accept_uniform<T>(a.rng.seed, (uint32_t)(a.rng.chain_offset + (uint64_t)m),
                                                          (uint32_t)a.rng.draw_offset, a.D)
                               : ln.uniform(a.rng, a.M, m, 0, 0));
            lu = __shfl_sync(0xffffffffu, lu, 0, G);
        }
        T ll_s, pr_s;
        if (!carry) md.terms(th, ll_c, pr_c);       // first step / replaced particles: nothing carried yet
        const T lp_c = A::add(A::mul(ll_c, t0), pr_c);
        bool acc;
        if constexpr (MOVE == BK_SMC_KERNEL_RW) {
#pragma unroll
            for (int k = 0; k < NE; ++k) st[k] = A::add(th[k], A::mul(a.scale, z[k]));  // smc.py:81
            md.terms(st, ll_s, pr_s);
            const T lp_s = A::add(A::mul(ll_s, t0), pr_s);
            acc = lu < A::sub(lp_s, lp_c);  // smc.py:85
        } else if constexpr (MOVE == BK_SMC_KERNEL_MALA) {
            // one MALA transition on the tempered density (mala.py:40-66)
            const T eps = a.scale, sd = A::sqrt_(A::mul(T(2), eps)), coef = T(-0.25) / eps;
#pragma unroll
            for (int k = 0; k < NE; ++k)
                st[k] = ln.valid(k) ? A::add(A::add(th[k], A::mul(eps, tgrad(th, k))), A::mul(sd, z[k])) : T(0);
            md.terms(st, ll_s, pr_s);
            const T lp_s = A::add(A::mul(ll_s, t0), pr_s);
            T sf = T(0), sr = T(0);
#pragma unroll
            for (int k = 0; k < NE; ++k) {
                if (ln.valid(k)) {
                    const T df = A::sub(A::sub(st[k], th[k]), A::mul(eps, tgrad(th, k)));
                    const T dr = A::sub(A::sub(th[k], st[k]), A::mul(eps, tgrad(st, k)));
                    sf = A::add(sf, A::mul(df, df));
                    sr = A::add(sr, A::mul(dr, dr));
                }
            }
            const T fwd = A::mul(coef, group_sum<G>(sf)), rev = A::mul(coef, group_sum<G>(sr));
            acc = lu < A::add(A::sub(lp_s, lp_c), A::sub(rev, fwd));   // metropolis.py:41-76
        } else {
            // one HMCDiag transition, identity metric, on the tempered density (hmc.py:40-63)
            const T eps = a.scale, heps = A::mul(T(0.5), eps);
            T kin = T(0);
#pragma unroll
            for (int k = 0; k < NE; ++k) kin = A::add(kin, A::mul(z[k], z[k]));
            const T h0 = A::sub(lp_c, A::mul(T(0.5), group_sum<G>(kin)));
#pragma unroll
            for (int k = 0; k < NE; ++k) {   // backward half kick (hmc.py:46)
                st[k] = th[k];
                z[k] = ln.valid(k) ? A::sub(z[k], A::mul(heps, tgrad(th, k))) : T(0);
            }
            for (int s = 0; s < a.steps; ++s) {   // hmc.py:47-50
#pragma unroll
                for (int k = 0; k < NE; ++k) {
                    if (ln.valid(k)) {
                        z[k] = A::add(z[k], A::mul(eps, tgrad(st, k)));
                        st[k] = A::add(st[k], A::mul(eps, z[k]));
                    }
                }
            }
            kin = T(0);
#pragma unroll
            for (int k = 0; k < NE; ++k) {   // forward half kick (hmc.py:52)
                if (ln.valid(k)) z[k] = A::add(z[k], A::mul(heps, tgrad(st, k)));
                kin = A::add(kin, A::mul(z[k], z[k]));
            }
            md.terms(st, ll_s, pr_s);
            const T h1 = A::sub(A::add(A::mul(ll_s, t0), pr_s), A::mul(T(0.5), group_sum<G>(kin)));
            acc = lu < A::sub(h1, h0);   // hmc.py:60
        }
        if (acc) {
#pragma unroll
            for (int k = 0; k < NE; ++k) th[k] = st[k];
            ll_c = ll_s;
            pr_c = pr_s;
        }
        // importance log-weight, both tempered densities in full (smc.py:67-70)
        const T lw = A::sub(A::add(A::mul(ll_c, a.t1), pr_c), A::add(A::mul(ll_c, a.t0), pr_c));
        if (active) {
            ln.store(a.thetas + m * (int64_t)a.D, th);
            if (ln.lane == 0) {
                if (a.llpr_out) { a.llpr_out[2 * m] = ll_c; a.llpr_out[2 * m + 1] = pr_c; }
                const T lw_tot = a.logw_prev ? A::add(a.logw_prev[m], lw) : lw;
                a.logw[m] = lw_tot;
                lw_max = fmax(lw_max, (double)lw_tot);
                if (a.accept) a.accept[m] = acc ? 1 : 0;
            }
        }
    }
    // statistics epilogue: the local maximum of the log-weights leaves with this launch -- the last CTA
    // to finish reduces the per-CTA maxima and posts (max, epoch) into every rank's mailbox
    if (a.maxpart) {
        __shared__ double red[33];
        __shared__ bool last_s;
        double v = warp_max(lw_max);
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane == 0) red[w] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int i = 1; i < (int)(blockDim.x >> 5); ++i) v = fmax(v, red[i]);
            a.maxpart[blockIdx.x] = v;
            __threadfence();
            last_s = atomicInc(a.ticket, gridDim.x - 1) == gridDim.x - 1;   // wraps to 0: self-resetting
        }
        __syncthreads();
        if (last_s) {
            __threadfence();
            double m2 = -INFINITY;
            for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) m2 = fmax(m2, ld_relaxed_gpu_f64(a.maxpart + i));
            m2 = warp_max(m2);
            __syncthreads();
            if (lane == 0) red[w] = m2;
            __syncthreads();
            if (threadIdx.x == 0) {
                for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m2 = fmax(m2, red[i]);
                red[32] = m2;
            }
            __syncthreads();
            const int nw = a.sh.world > 0 ? a.sh.world : 1;
            if ((int)threadIdx.x < nw)
                mail_post1(a.mail_tab[threadIdx.x] + MB_MAX + ((a.epoch & 1) * BK_SMC_MAX_WORLD + a.sh.rank) * 2,
                           (uint64_t)__double_as_longlong(red[32]), a.epoch);
        }
    }
}

static int device_sms() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

template <typename T, int G, int J, template <typename, int, int> class View, int MOVE, int OCC = 0, int VM = -1>
static int launch_smc3(const SmcArgs<T>& a, cudaStream_t st) {
    const int64_t per_block = 128 / G;
    const int64_t need = (a.M + per_block - 1) / per_block;
    // persistent: exactly one wave -- as many CTAs of 128 threads as are resident at once (8 per SM at 62
    // registers, 3 for the 16-elements-per-lane layout); every B200 of a box has the same SM count
    static int64_t cap = 0;
    if (!cap) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_smc_move_weight<T, G, J, View, MOVE, OCC, VM>, 128, 0) != cudaSuccess || nb < 1) {
            cudaGetLastError();
            nb = 1;
        }
        cap = (int64_t)device_sms() * (nb > 8 ? 8 : nb);
    }
    int64_t blocks = need < cap ? need : cap;
    if (blocks > SMC_MAXPART) blocks = SMC_MAXPART;
    k_smc_move_weight<T, G, J, View, MOVE, OCC, VM><<<(unsigned)blocks, 128, 0, st>>>(a);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

template <typename T, int G, int J, template <typename, int, int> class View>
static int launch_smc(const SmcArgs<T>& a, int move, cudaStream_t st) {
    switch (move) {
        case BK_SMC_KERNEL_RW: return launch_smc3<T, G, J, View, BK_SMC_KERNEL_RW>(a, st);
        case BK_SMC_KERNEL_MALA: return launch_smc3<T, G, J, View, BK_SMC_KERNEL_MALA>(a, st);
        case BK_SMC_KERNEL_HMC: return launch_smc3<T, G, J, View, BK_SMC_KERNEL_HMC>(a, st);
    }
    set_error("unknown SMC kernel kind %d", move);
    return BK_E_INVALID;
}

// a prior/likelihood user model: the same arguments, as the plain fields of its runtime-compiled kernel
template <typename T>
static int smc_user(const Model& m, const SmcArgs<T>& a, const bk_smc_kernel& kn, cudaStream_t st) {
    UserSmcArgs u;
    memset(&u, 0, sizeof(u));
    u.thetas = a.thetas;
    u.src = a.src;
    u.src_idx = a.src_idx;
    u.M = a.M;
    u.t0 = (double)a.t0;
    u.t1 = (double)a.t1;
    u.scale = kn.scale;
    u.steps = kn.steps;
    u.rng_mode = a.rng.mode;
    u.n_uniform = a.rng.n_uniform;
    u.seed = a.rng.seed;
    u.draw_offset = a.rng.draw_offset;
    u.chain_offset = a.rng.chain_offset;
    u.normals = a.rng.normals;
    u.uniforms = a.rng.uniforms;
    u.logw = a.logw;
    u.logw_prev = a.logw_prev;
    u.accept = a.accept;
    u.sh = a.sh;
    for (int r = 0; r < BK_SMC_MAX_WORLD; ++r) {
        u.src_tab[r] = a.src_tab[r];
        u.llpr_tab[r] = a.llpr_tab[r];
        u.mail_tab[r] = a.mail_tab[r];
    }
    u.llpr_out = a.llpr_out;
    u.carry = a.carry;
    u.epoch = a.epoch;
    u.wait_done = a.wait_done;
    u.maxpart = a.maxpart;
    u.ticket = a.ticket;
    u.params = m.user_params;
    const UserProposal* p = nullptr;
    if (kn.kind == BK_SMC_KERNEL_PROPOSAL) {   // check_smc_model resolved the handle
        p = get_proposal(kn.proposal);
        if (!p) return BK_E_HANDLE;
        u.prop_params = p->params;
    }
    return user_smc_move(m, p, kn.kind, u, st);
}

// fills the model / geometry part of the arguments and picks the lane layout
template <typename T>
static int smc_dispatch(const Model& m, SmcArgs<T>& a, const bk_smc_kernel& kn, cudaStream_t st) {
    if (m.d.kind == BK_MODEL_USER_CUDA) return smc_user<T>(m, a, kn, st);
    a.D = (int)m.d.dims;
    a.scale = (T)kn.scale;
    a.steps = kn.steps;
    if (m.d.kind == BK_MODEL_BINOMIAL_LOGIT) {
        for (int i = 0; i < 6; ++i) a.bp[i] = (T)m.d.scalars[i];
        a.vec = a.vec2 = 0;
        return launch_smc<T, 1, 1, BinomView>(a, kn.kind, st);
    }
    a.mu = (const T*)m.d.mu; a.pl = (const T*)m.d.prec; a.m0 = (const T*)m.d.m0; a.p0 = (const T*)m.d.p0;
    auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    bool tabs16 = true, tabs8 = true;
    auto al8 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7) == 0; };
    for (int r = 0; r < a.sh.world; ++r) { tabs16 = tabs16 && al(a.src_tab[r]); tabs8 = tabs8 && al8(a.src_tab[r]); }
    a.vec = (a.D % 4 == 0 && al(a.thetas) && al(a.src) && tabs16 && al(a.mu) && al(a.pl) && al(a.m0) && al(a.p0) &&
             (a.rng.mode != BK_RNG_INJECTED || al(a.rng.normals))) ? 1 : 0;
    // D even but not a multiple of 4 (c4: D = 50): rows are 8-byte aligned -> 64-bit accesses
    a.vec2 = (!a.vec && sizeof(T) == 4 && a.D % 2 == 0 && al8(a.thetas) && al8(a.src) && tabs8 && al8(a.mu) && al8(a.pl) &&
              al8(a.m0) && al8(a.p0) && (a.rng.mode != BK_RNG_INJECTED || al8(a.rng.normals))) ? 1 : 0;
    const int D = a.D;
    if (D <= 4) return launch_smc<T, 1, 1, GplView>(a, kn.kind, st);
    if (D <= 16) return launch_smc<T, 4, 1, GplView>(a, kn.kind, st);
    if (D <= 32) return launch_smc<T, 8, 1, GplView>(a, kn.kind, st);
    // fp32 (timed mode), RW move: 4 lanes x 16 elements instead of 16 x 4 -- the per-lane overhead of a particle visit
    // is paid by a quarter of the lanes; G * J (Philox blocks, spare-block uniform rule) is unchanged.  BK_SEP_WIDE=0: off
    static int wide = -1;
    if (wide < 0) { const char* e = getenv("BK_SEP_WIDE"); wide = (e && e[0] == '0') ? 0 : 1; }
    if constexpr (sizeof(T) == 4) {
        static int layout = -1;   // BK_SMC_LAYOUT (diagnostic): 2 = 4 x 16 (default), 1 = 8 x 8, 0 = 16 x 4
        if (layout < 0) { const char* e = getenv("BK_SMC_LAYOUT"); layout = e ? atoi(e) : 2; }
        if (wide && D > 32 && D <= 64 && kn.kind == BK_SMC_KERNEL_RW) {
            static int occ = -1;
            if (occ < 0) { const char* e = getenv("BK_SMC_OCC"); occ = e ? atoi(e) : 0; }
            if (layout == 2 && occ == 2) return launch_smc3<T, 4, 4, GplView, BK_SMC_KERNEL_RW, 2>(a, st);
            if (layout == 2 && occ == 4) return launch_smc3<T, 4, 4, GplView, BK_SMC_KERNEL_RW, 4>(a, st);
            if (layout == 2 && a.vec) return launch_smc3<T, 4, 4, GplView, BK_SMC_KERNEL_RW, 0, 1>(a, st);
            if (layout == 2 && a.vec2) return launch_smc3<T, 4, 4, GplView, BK_SMC_KERNEL_RW, 0, 2>(a, st);
            if (layout == 2) return launch_smc3<T, 4, 4, GplView, BK_SMC_KERNEL_RW>(a, st);
            if (layout == 1) return launch_smc3<T, 8, 2, GplView, BK_SMC_KERNEL_RW>(a, st);
        }
    }
    if (D <= 64) return launch_smc<T, 16, 1, GplView>(a, kn.kind, st);
    if (D <= 128) return launch_smc<T, 32, 1, GplView>(a, kn.kind, st);
    if (D <= 256) return launch_smc<T, 32, 2, GplView>(a, kn.kind, st);
    set_error("bk_smc_move_weight supports D <= 256 (got %d)", D);
    return BK_E_UNSUPPORTED;
}

// the PROPOSAL kind: a user prior/likelihood model and a proposal of its dims and dtype; rng (may be NULL): the
// injected uniforms carry the accept uniform and the proposal's
static int check_smc_proposal(const Model& m, const bk_smc_kernel& kn, const bk_rng* rng) {
    if (!user_prior_lik(m)) {
        set_error("bk_smc: the proposal move runs on user models created by bk_model_create_cuda_prior_lik only "
                  "(restate a built-in GAUSS_PRIOR_LIK / BINOMIAL_LOGIT model as one)");
        return BK_E_UNSUPPORTED;
    }
    const UserProposal* p = get_proposal(kn.proposal);
    if (!p) return BK_E_HANDLE;
    BK_CHECK_ARG(m.d.dims == p->dims && m.d.dtype == p->dtype,
                 "bk_smc: the proposal (dims %lld, dtype %d) does not match the model (dims %lld, dtype %d)",
                 (long long)p->dims, p->dtype, (long long)m.d.dims, m.d.dtype);
    BK_CHECK_ARG(p->n_normals <= BK_SMC_PROPOSAL_MAX_NORMALS,
                 "bk_smc: the proposal move supports n_normals <= %d (got %d)", BK_SMC_PROPOSAL_MAX_NORMALS,
                 p->n_normals);
    BK_CHECK_ARG(!rng || rng->mode != BK_RNG_INJECTED || rng->n_uniform == 1 + p->n_uniforms,
                 "bk_smc: injected rng needs n_uniform = 1 + the proposal's n_uniforms = %d (got %d)",
                 1 + p->n_uniforms, rng ? rng->n_uniform : 0);
    return BK_OK;
}

static int check_smc_model(const Model& m, const bk_smc_kernel& kn, const bk_rng* rng = nullptr) {
    BK_CHECK_ARG(m.d.kind == BK_MODEL_GAUSS_PRIOR_LIK || m.d.kind == BK_MODEL_BINOMIAL_LOGIT || user_prior_lik(m),
                 "bk_smc_move_weight: the model must expose log_prior / log_likelihood (GAUSS_PRIOR_LIK, BINOMIAL_LOGIT, "
                 "or a user model created by bk_model_create_cuda_prior_lik)");
    BK_CHECK_ARG(m.d.kind != BK_MODEL_USER_CUDA || m.d.dims <= BK_USER_PRIOR_LIK_MAX_DIMS,
                 "bk_smc_move_weight: user models support dims <= %d (got %lld)", BK_USER_PRIOR_LIK_MAX_DIMS,
                 (long long)m.d.dims);
    BK_CHECK_ARG(kn.kind >= BK_SMC_KERNEL_RW && kn.kind <= BK_SMC_KERNEL_PROPOSAL, "bk_smc: unknown kernel kind %d",
                 kn.kind);
    if (kn.kind == BK_SMC_KERNEL_PROPOSAL) return check_smc_proposal(m, kn, rng);
    BK_CHECK_ARG(kn.scale > 0, "bk_smc: kernel scale / step size must be positive (got %g)", kn.scale);
    BK_CHECK_ARG(kn.kind != BK_SMC_KERNEL_HMC || kn.steps >= 0, "bk_smc: HMC kernel needs steps >= 0");
    return BK_OK;
}

template <typename T>
static int smc_move_t(const Model& m, const void* src, const int64_t* src_idx, void* thetas, int64_t M,
                      int n, int Tn, const bk_smc_kernel& kn, const bk_rng* rng, void* logw, const void* logw_prev,
                      int32_t* accept, cudaStream_t st) {
    SmcArgs<T> a;
    memset(&a, 0, sizeof(a));
    a.thetas = (T*)thetas;
    a.src = (const T*)src;
    a.src_idx = src_idx;
    a.M = M;
    a.t0 = (T)((double)(n - 1) / Tn);  // smc.py:43-44
    a.t1 = (T)((double)n / Tn);
    a.rng = *rng;
    a.logw = (T*)logw;
    a.logw_prev = (const T*)logw_prev;
    a.accept = accept;
    return smc_dispatch<T>(m, a, kn, st);
}

// ---- weight statistics ---------------------------------------------------------
constexpr int RED_THREADS = 256;

template <typename T>
__global__ void k_max_partial(const T* __restrict__ x, int64_t n, double* __restrict__ part) {
    __shared__ double sm[33];
    double v = -INFINITY;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        v = fmax(v, (double)x[i]);
    v = warp_max(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) sm[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < (blockDim.x >> 5) ? sm[lane] : -INFINITY;
        v = warp_max(v);
        if (lane == 0) part[blockIdx.x] = v;
    }
}

// single block: out[0] = max over the block partials (0 when the weights are not shifted)
__global__ void k_max_final(const double* __restrict__ maxpart, int nb, int use_shift, double* __restrict__ out) {
    __shared__ double sm[33];
    double v = -INFINITY;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) v = fmax(v, maxpart[i]);
    v = warp_max(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) sm[w] = v;
    __syncthreads();
    if (w == 0) {
        v = lane < (blockDim.x >> 5) ? sm[lane] : -INFINITY;
        v = warp_max(v);
        if (lane == 0) out[0] = use_shift ? v : 0.0;
    }
}

// per-block sums of exp(x - shift) and its square, shift = stats[0]
template <typename T>
__global__ void k_sum_partial(const T* __restrict__ x, int64_t n, const double* __restrict__ stats,
                              double* __restrict__ part) {
    __shared__ double sm[33];
    const double shift = stats[0];
    double s = 0, s2 = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double w = exp((double)x[i] - shift);
        s += w;
        s2 += w * w;
    }
    s = block_sum(s, sm);
    s2 = block_sum(s2, sm);
    if (threadIdx.x == 0) {
        part[2 * blockIdx.x] = s;
        part[2 * blockIdx.x + 1] = s2;
    }
}

// single block, fixed order: out[1] = sum w, out[2] = sum w^2
__global__ void k_stats_final(const double* __restrict__ part, int nb, double* __restrict__ out) {
    __shared__ double sm[33];
    double s = 0, s2 = 0;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) {
        s += part[2 * i];
        s2 += part[2 * i + 1];
    }
    s = block_sum(s, sm);
    s2 = block_sum(s2, sm);
    if (threadIdx.x == 0) {
        out[1] = s;
        out[2] = s2;
    }
}

// ---- CDF: p_i = exp(logw_i - shift) / total ; inclusive scan ; cdf /= cdf[-1] ----
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 4, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename T>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_local(const T* __restrict__ logw, int64_t n,
                                                             double shift, double total,
                                                             const double* __restrict__ stats, int mode,
                                                             double* __restrict__ cdf,
                                                             double* __restrict__ block_tot) {
    __shared__ double wsum[SCAN_THREADS / 32];
    if (stats) {  // normaliser produced on device by bk_smc_weight_stats
        shift = stats[0];
        total = mode == BK_RESAMPLE_MULTINOMIAL ? stats[1] : 1.0;
    }
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    double v[SCAN_ITEMS];
    double run = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        int64_t j = base + i;
        double w = j < n ? exp((double)logw[j] - shift) / total : 0.0;
        run += w;
        v[i] = run;
    }
    // inclusive scan of per-thread totals
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        double t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    double woff = 0;
    for (int i = 0; i < w; ++i) woff += wsum[i];
    const double excl = woff + inc - run;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        int64_t j = base + i;
        if (j < n) cdf[j] = excl + v[i];
    }
    if (threadIdx.x == SCAN_THREADS - 1) block_tot[blockIdx.x] = excl + run;
}

// exclusive scan of the block totals: one CTA of 1024 threads walks chunks of 1024 totals
__global__ void __launch_bounds__(1024) k_scan_blocks(double* __restrict__ block_tot, int nb,
                                                      double* __restrict__ grand) {
    __shared__ double wsum[32];
    __shared__ double carry_s;
    if (threadIdx.x == 0) carry_s = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int base = 0; base < nb; base += 1024) {
        const int i = base + threadIdx.x;
        const double v = i < nb ? block_tot[i] : 0.0;
        double inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            double t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) wsum[w] = inc;
        __syncthreads();
        double woff = 0;
        for (int k = 0; k < w; ++k) woff += wsum[k];
        const double carry = carry_s;
        if (i < nb) block_tot[i] = carry + woff + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + woff + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) *grand = carry_s;
}

__global__ void k_scan_finish(double* __restrict__ cdf, int64_t n, const double* __restrict__ block_off,
                              const double* __restrict__ grand) {
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    // cdf /= cdf[-1]  (legacy choice, SURVEY.md 2.1-9)
    cdf[j] = (cdf[j] + block_off[j / SCAN_TILE]) / *grand;
}

template <typename T>
__global__ void k_search(const double* __restrict__ cdf, int64_t M, int mode, const T* __restrict__ u_in,
                         bk_rng rng, int64_t n_points, int64_t point_offset,
                         int64_t* __restrict__ idx) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_points) return;
    double u;
    if (mode == BK_RESAMPLE_MULTINOMIAL) {
        u = u_in ? (double)u_in[i]
                 : (double)philox_uniform<T>(rng.seed, 0, (uint32_t)(point_offset + i),
                                             (uint32_t)rng.draw_offset, TAG_RESAMPLE);
    } else {
        double u0 = u_in ? (double)u_in[0]
                         : (double)philox_uniform<T>(rng.seed, 0, 0u, (uint32_t)rng.draw_offset, TAG_RESAMPLE);
        u = ((double)(point_offset + i) + u0) / (double)M;
    }
    // first index with cdf[idx] > u  (searchsorted side='right')
    int64_t lo = 0, hi = M;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (cdf[mid] <= u) lo = mid + 1;
        else hi = mid;
    }
    idx[i] = lo < M ? lo : M - 1;
}

template <typename T>
__global__ void k_gather(const T* __restrict__ src, const int64_t* __restrict__ idx, int64_t M, int D,
                         T* __restrict__ out) {
    int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (r >= M) return;
    const T* s = src + idx[r] * (int64_t)D;
    T* o = out + r * (int64_t)D;
    for (int e = lane; e < D; e += 32) o[e] = s[e];
}

// Adaptive resampling: resample only when the importance-weight ESS (sum w)^2 / sum w^2 falls below
// the threshold; otherwise the particles stay (identity indices) and keep their log-weights.  The
// decision is taken on device from the stats bk_smc_weight_stats wrote -- no host round trip.
template <typename T>
__global__ void k_smc_adaptive_select(const double* __restrict__ stats, double thr, int64_t n, int64_t point_offset,
                                      int64_t* __restrict__ idx, T* __restrict__ logw, int32_t* __restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool resample = stats[1] * stats[1] / stats[2] < thr;
    if (i == 0 && flag) *flag = resample ? 1 : 0;
    if (i >= n) return;
    if (resample) logw[i] = T(0);            // equal weights after resampling
    else idx[i] = point_offset + i;          // keep particle i and its accumulated log-weight
}


// =====================================================================================
// Sharded resampling (bk_smc_shard_*): fixed-point systematic resampling in two kernels,
// cross-rank traffic through mailboxes / peer stores (smc_shard.cuh, bk.h)
// =====================================================================================
constexpr int SC_THREADS = 256, SC_ITEMS = 4, SC_TILE = SC_THREADS * SC_ITEMS;
constexpr int RS_POINTS = 8;      // consecutive systematic points resolved per thread

// control words at the head of the local workspace (zeroed once by the caller)
enum { CT_MOVE = 0, CT_SCAN_DONE = 2, CT_RES_DONE = 3, CT_WORDS = 16 };

struct ShardWs {
    unsigned* ctrl;      // [CT_WORDS]
    double* maxpart;     // [SMC_MAXPART]
    double* qpart;       // [n_tiles]
    int64_t* tile_off;   // [n_tiles + 1] tile totals, then (last CTA of the scan) their exclusive prefix; [n_tiles] = W
    int64_t* cum;        // [n_max]   inclusive cumsum of the fixed-point weights WITHIN each tile
    char* extra;         // multinomial: all log-weights [M] + the single-GPU resampler's scratch
    size_t extra_bytes;
    int64_t n_tiles;
};
static int64_t shard_n_max(int64_t M, int world) { return (M + world - 1) / world; }
static size_t shard_ws_layout(void* ws, size_t ws_bytes, int64_t M, int world, ShardWs* out) {
    Arena ar(ws, ws_bytes);
    const int64_t n_max = shard_n_max(M, world), n_tiles = (n_max + SC_TILE - 1) / SC_TILE;
    ShardWs w;
    w.ctrl = ar.take<unsigned>(CT_WORDS);
    w.maxpart = ar.take<double>(SMC_MAXPART);
    w.qpart = ar.take<double>(n_tiles);
    w.tile_off = ar.take<int64_t>(n_tiles + 1);
    w.cum = ar.take<int64_t>(n_max);
    w.extra = ar.take<char>(0);
    w.extra_bytes = ws_bytes > ar.off ? ws_bytes - ar.off : 0;
    w.n_tiles = n_tiles;
    if (out) *out = w;
    return ar.off;
}

struct ScanArgs {
    const void* logw;       // [n] local log-weights (dtype)
    int64_t n;              // local particle count
    int shift_bits;         // s: w = rint(exp(logw - gmax) * 2^s)
    ShardGeom sh;
    uint64_t* mail_tab[BK_SMC_MAX_WORLD];
    uint64_t epoch;
    int64_t* cum;
    int64_t* tile_off;
    double* qpart;
    unsigned* ctrl;
    int64_t n_tiles;
};

__device__ __forceinline__ int64_t fixed_weight(double lw, double gmax, int s) {
    const double e = exp(lw - gmax);
    return e == e ? __double2ll_rn(ldexp(e, s)) : 0;   // NaN log-weight: no mass
}

// One CTA per tile of 1024 particles: fixed-point weights, inclusive scan within the tile, tile total.
// The last CTA to finish turns the tile totals into their exclusive prefix (one CTA, integer adds: a few
// microseconds for thousands of tiles) and posts the local mass W and sum of squares Q to every rank.
template <typename T>
__global__ void __launch_bounds__(SC_THREADS) k_smc_scan(ScanArgs a) {
    __shared__ double gmax_s;
    __shared__ int64_t wsum[SC_THREADS / 32];
    __shared__ double qred[33];
    __shared__ bool last_s;
    __shared__ int64_t carry_s;
    uint64_t* mine = a.mail_tab[a.sh.rank];
    if (threadIdx.x < 32) {   // global max of the log-weights from the G max messages
        double v = -INFINITY;
        if ((int)threadIdx.x < a.sh.world) {
            const uint64_t* slot = mine + MB_MAX + ((a.epoch & 1) * BK_SMC_MAX_WORLD + threadIdx.x) * 2;
            mail_wait(slot + 1, a.epoch, mine);
            v = __longlong_as_double((long long)ld_relaxed_sys(slot));
        }
        v = warp_max(v);
        if (threadIdx.x == 0) gmax_s = v;
    }
    __syncthreads();
    const double gmax = gmax_s;
    const int64_t tile = blockIdx.x;
    const T* lw = (const T*)a.logw;
    const int64_t base = tile * SC_TILE + (int64_t)threadIdx.x * SC_ITEMS;
    int64_t v[SC_ITEMS], run = 0;
    double q = 0.0;
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i) {
        const int64_t j = base + i;
        const int64_t w = j < a.n ? fixed_weight((double)lw[j], gmax, a.shift_bits) : 0;
        run += w;
        v[i] = run;
        const double wd = (double)w;
        q += wd * wd;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[wid] = inc;
    q = warp_sum(q);
    if (lane == 0) qred[wid] = q;
    __syncthreads();
    int64_t woff = 0, agg = 0;
#pragma unroll
    for (int i = 0; i < SC_THREADS / 32; ++i) {
        if (i < wid) woff += wsum[i];
        agg += wsum[i];
    }
    const int64_t excl = woff + inc - run;
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i) {
        const int64_t j = base + i;
        if (j < a.n) a.cum[j] = excl + v[i];
    }
    if (threadIdx.x == 0) {
        double qs = 0.0;
        for (int i = 0; i < SC_THREADS / 32; ++i) qs += qred[i];   // fixed order
        a.qpart[tile] = qs;
        a.tile_off[tile] = agg;
        __threadfence();
        last_s = atomicInc(a.ctrl + CT_SCAN_DONE, gridDim.x - 1) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last_s) return;
    __threadfence();
    // exclusive prefix of the tile totals, SC_THREADS tiles per round
    if (threadIdx.x == 0) carry_s = 0;
    double qs = 0.0;
    __syncthreads();
    for (int64_t t0 = 0; t0 < a.n_tiles; t0 += SC_THREADS) {
        const int64_t t = t0 + threadIdx.x;
        const int64_t x = t < a.n_tiles ? (int64_t)ld_relaxed_gpu((const uint64_t*)a.tile_off + t) : 0;
        if (t < a.n_tiles) qs += ld_relaxed_gpu_f64(a.qpart + t);
        int64_t in2 = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, in2, o);
            if (lane >= o) in2 += y;
        }
        if (lane == 31) wsum[wid] = in2;
        __syncthreads();
        int64_t wo = 0, tot = 0;
#pragma unroll
        for (int i = 0; i < SC_THREADS / 32; ++i) {
            if (i < wid) wo += wsum[i];
            tot += wsum[i];
        }
        const int64_t carry = carry_s;
        if (t < a.n_tiles) a.tile_off[t] = carry + wo + in2 - x;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
    qs = warp_sum(qs);
    if (lane == 0) qred[wid] = qs;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < SC_THREADS / 32; ++i) t += qred[i];
        qred[32] = t;
        a.tile_off[a.n_tiles] = carry_s;
    }
    __syncthreads();
    if ((int)threadIdx.x < a.sh.world)
        mail_post3(a.mail_tab[threadIdx.x] + MB_MASS + ((a.epoch & 1) * BK_SMC_MAX_WORLD + a.sh.rank) * 4, (uint64_t)carry_s,
                   (uint64_t)__double_as_longlong(qred[32]), (uint64_t)a.n, a.epoch);
}

struct ResolveArgs {
    ShardGeom sh;
    uint64_t* mail_tab[BK_SMC_MAX_WORLD];
    int64_t* idx_tab[BK_SMC_MAX_WORLD];
    uint64_t epoch;
    const int64_t* cum;     // inclusive cumsum within each tile [n]
    const int64_t* tile_off;  // exclusive prefix of the tile totals [n_tiles]
    int64_t n, n_tiles;
    int shift_bits;
    const void* u0_in;      // injected u0 (dtype) or NULL
    bk_rng rng;
    double ess_threshold;   // > 0: adaptive
    void* logw;             // local log-weights (zeroed when an adaptive step resamples)
    double* stats_out;      // [4] or NULL
    unsigned* ctrl;
};

// threshold of systematic point k in fixed-point CDF units: floor((k + u0) * (W / M)), clamped below W
// (fp64 operations in this order; `rate` = (double)W / (double)M is formed once)
__device__ __forceinline__ int64_t sys_threshold(int64_t k, double u0, double rate, int64_t W) {
    const int64_t ti = (int64_t)floor(__dmul_rn(__dadd_rn((double)k, u0), rate));
    return ti < W ? ti : W - 1;
}

constexpr int RS_SMEM_TILES = 4096;   // tile offsets cached in shared memory (32 KB): 4 M particles per rank

template <typename T>
__global__ void __launch_bounds__(256) k_smc_resolve(ResolveArgs a) {
    __shared__ int64_t Ws[BK_SMC_MAX_WORLD];
    __shared__ double Qs[BK_SMC_MAX_WORLD];
    __shared__ int64_t k_lo_s, k_hi_s, off_s, tot_s;
    __shared__ double u0_s;
    __shared__ int resample_s;
    __shared__ bool last_s;
    __shared__ int64_t toff_s[RS_SMEM_TILES];
    uint64_t* mine = a.mail_tab[a.sh.rank];
    if ((int)threadIdx.x < a.sh.world) {
        const uint64_t* slot = mine + MB_MASS + ((a.epoch & 1) * BK_SMC_MAX_WORLD + threadIdx.x) * 4;
        mail_wait(slot + 3, a.epoch, mine);
        Ws[threadIdx.x] = (int64_t)ld_relaxed_sys(slot);
        Qs[threadIdx.x] = __longlong_as_double((long long)ld_relaxed_sys(slot + 1));
    }
    const bool toff_in_smem = a.n_tiles <= RS_SMEM_TILES;
    if (toff_in_smem)
        for (int64_t i = threadIdx.x; i < a.n_tiles; i += blockDim.x) toff_s[i] = a.tile_off[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t off = 0, tot = 0;
        double q = 0.0;
        for (int r = 0; r < a.sh.world; ++r) {   // rank order on every rank: identical decisions
            if (r < a.sh.rank) off += Ws[r];
            tot += Ws[r];
            q += Qs[r];
        }
        const double u0 = a.u0_in ? (double)((const T*)a.u0_in)[0]
                                  : (double)philox_uniform<T>(a.rng.seed, 0, 0u, (uint32_t)a.rng.draw_offset, TAG_RESAMPLE);
        const double Wd = (double)tot, rate = Wd / (double)a.sh.M;
        int resample = 1;
        if (a.ess_threshold > 0) resample = (Wd * Wd / q < a.ess_threshold) ? 1 : 0;
        if (tot <= 0) { resample = 0; st_relaxed_sys(mine + MB_ERR, 2ull); }   // every weight vanished: keep the particles
        // first point whose threshold reaches `target` (thresholds are monotone in k): estimate, then fix up
        auto first_at = [&](int64_t target) {
            if (target <= 0) return (int64_t)0;
            int64_t lo = 0, hi = a.sh.M;
            const double guess = (double)target / rate - u0;
            int64_t g = (int64_t)guess;
            if (g > 4 && g < a.sh.M - 4) {        // narrow the bracket around the estimate when it is consistent
                if (sys_threshold(g - 4, u0, rate, tot) < target) lo = g - 4;
                if (sys_threshold(g + 4, u0, rate, tot) >= target) hi = g + 4;
            }
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (sys_threshold(mid, u0, rate, tot) < target) lo = mid + 1; else hi = mid;
            }
            return lo;
        };
        k_lo_s = resample ? first_at(off) : 0;
        k_hi_s = resample ? (a.sh.rank == a.sh.world - 1 ? a.sh.M : first_at(off + Ws[a.sh.rank])) : 0;
        off_s = off; tot_s = tot; u0_s = u0; resample_s = resample;
        if (blockIdx.x == 0 && a.stats_out) {
            double mx = -INFINITY;
            for (int r = 0; r < a.sh.world; ++r)
                mx = fmax(mx, __longlong_as_double((long long)ld_relaxed_sys(mine + MB_MAX + ((a.epoch & 1) * BK_SMC_MAX_WORLD + r) * 2)));
            a.stats_out[0] = mx;
            a.stats_out[1] = ldexp(Wd, -a.shift_bits);
            a.stats_out[2] = ldexp(q, -2 * a.shift_bits);
            a.stats_out[3] = (double)resample;
        }
    }
    __syncthreads();
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gstride = (int64_t)gridDim.x * blockDim.x;
    const int64_t lo_r = shard_lo(a.sh, a.sh.rank);
    if (resample_s) {
        const int64_t k_lo = k_lo_s, k_hi = k_hi_s, off = off_s, tot = tot_s;
        const double u0 = u0_s, rate = (double)tot / (double)a.sh.M;
        const int64_t* toff = toff_in_smem ? toff_s : a.tile_off;
        // a thread resolves RS_POINTS consecutive points: one two-level search (tile offsets, then inside the
        // tile) for the first, a short forward walk for the others (consecutive points sit ~1 particle apart)
        for (int64_t k0 = k_lo + gtid * RS_POINTS; k0 < k_hi; k0 += gstride * RS_POINTS) {
            int64_t t = sys_threshold(k0, u0, rate, tot) - off;          // in [0, W_r)
            int64_t tl = 0, th = a.n_tiles;                              // last tile with toff <= t
            while (th - tl > 1) {
                const int64_t mid = (tl + th) >> 1;
                if (toff[mid] <= t) tl = mid; else th = mid;
            }
            int64_t tile = tl, tbase = toff[tile];
            int64_t jend = (tile + 1) * SC_TILE < a.n ? (tile + 1) * SC_TILE : a.n;
            int64_t lo = tile * SC_TILE, hi = jend;                      // first j in the tile with cum[j] > t - tbase
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (a.cum[mid] <= t - tbase) lo = mid + 1; else hi = mid;
            }
            int64_t j = lo;
#pragma unroll 1
            for (int p = 0; p < RS_POINTS; ++p) {
                const int64_t k = k0 + p;
                if (k >= k_hi) break;
                if (p > 0) {
                    t = sys_threshold(k, u0, rate, tot) - off;
                    // advance to the first particle whose global inclusive cumsum exceeds t
                    while (true) {
                        if (j >= jend) {                                   // tile exhausted: next tile with mass
                            if (jend >= a.n) { j = a.n - 1; break; }
                            ++tile; tbase = toff[tile];
                            jend = (tile + 1) * SC_TILE < a.n ? (tile + 1) * SC_TILE : a.n;
                            j = tile * SC_TILE;
                            continue;
                        }
                        if (tbase + a.cum[j] > t) break;
                        ++j;
                    }
                } else if (j >= jend) {
                    // t falls on a tile whose remaining particles carry no mass beyond it (cannot happen when
                    // toff[tile + 1] > t, which the tile search guarantees) -- clamp defensively
                    j = jend - 1;
                }
                int owner; int64_t loc;
                shard_locate(a.sh, k, owner, loc);
                a.idx_tab[owner][loc] = lo_r + j;     // peer store: the slot's owner reads it in its next move
            }
        }
        if (a.ess_threshold > 0)                   // equal weights after an adaptive step resampled
            for (int64_t i = gtid; i < a.n; i += gstride) ((T*)a.logw)[i] = T(0);
    } else {
        for (int64_t i = gtid; i < a.n; i += gstride) a.idx_tab[a.sh.rank][i] = lo_r + i;   // keep particle and weight
    }
    // done message once every CTA's index stores are out
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) last_s = atomicInc(a.ctrl + CT_RES_DONE, gridDim.x - 1) == gridDim.x - 1;
    __syncthreads();
    if (last_s) {
        __threadfence_system();
        if ((int)threadIdx.x < a.sh.world)
            st_release_sys(a.mail_tab[threadIdx.x] + MB_DONE + (a.epoch & 1) * BK_SMC_MAX_WORLD + a.sh.rank, a.epoch);
    }
}

// multinomial at world > 1: every rank copies all log-weights from its peers (after their max
// messages, i.e. after their move kernels) and runs the single-GPU fp64 CDF on the copy
struct CollectArgs {
    ShardGeom sh;
    uint64_t* mailbox;
    const void* logw_tab[BK_SMC_MAX_WORLD];
    uint64_t epoch;
    void* out;
};
template <typename T>
__global__ void k_smc_collect(CollectArgs a) {
    if ((int)threadIdx.x < a.sh.world)
        mail_wait(a.mailbox + MB_MAX + ((a.epoch & 1) * BK_SMC_MAX_WORLD + threadIdx.x) * 2 + 1, a.epoch, a.mailbox);
    __syncthreads();
    T* out = (T*)a.out;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < a.sh.M; g += (int64_t)gridDim.x * blockDim.x) {
        int r; int64_t loc;
        shard_locate(a.sh, g, r, loc);
        out[g] = ((const T*)a.logw_tab[r])[loc];
    }
}

struct DoneArgs {
    ShardGeom sh;
    uint64_t* mail_tab[BK_SMC_MAX_WORLD];
    uint64_t epoch;
};
__global__ void k_smc_post_done(DoneArgs a) {
    __threadfence_system();
    if ((int)threadIdx.x < a.sh.world)
        st_release_sys(a.mail_tab[threadIdx.x] + MB_DONE + (a.epoch & 1) * BK_SMC_MAX_WORLD + a.sh.rank, a.epoch);
}

struct GatherArgs {
    ShardGeom sh;
    uint64_t* mailbox;
    const void* src_tab[BK_SMC_MAX_WORLD];
    const int64_t* idx;
    uint64_t epoch;
    int64_t n;
    int D;
    void* out;
};
template <typename T>
__global__ void k_smc_gather_sharded(GatherArgs a) {
    if ((int)threadIdx.x < a.sh.world)
        mail_wait(a.mailbox + MB_DONE + (a.epoch & 1) * BK_SMC_MAX_WORLD + threadIdx.x, a.epoch, a.mailbox);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < a.n; r += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        int owner; int64_t loc;
        shard_locate(a.sh, a.idx[r], owner, loc);
        const T* s = (const T*)a.src_tab[owner] + loc * (int64_t)a.D;
        T* o = (T*)a.out + r * (int64_t)a.D;
        for (int e = lane; e < a.D; e += 32) o[e] = s[e];
    }
}

static int make_geom(const bk_smc_shard* sh, ShardGeom* g) {
    BK_CHECK_ARG(sh && sh->world >= 1 && sh->world <= BK_SMC_MAX_WORLD && sh->rank >= 0 && sh->rank < sh->world,
                 "bk_smc_shard: need 0 <= rank < world <= %d", BK_SMC_MAX_WORLD);
    BK_CHECK_ARG(sh->M >= sh->world, "bk_smc_shard: need at least one particle per rank (M=%lld, world=%d)",
                 (long long)sh->M, sh->world);
    BK_CHECK_ARG(sh->epoch >= 1, "bk_smc_shard: epoch counts from 1");
    g->world = sh->world;
    g->rank = sh->rank;
    g->M = sh->M;
    g->base = sh->M / sh->world;
    g->extra = (int32_t)(sh->M % sh->world);
    g->small = sh->M < (1ll << 32) ? 1 : 0;
    for (int r = 0; r < sh->world; ++r)
        BK_CHECK_ARG(sh->mailbox[r] && sh->logw[r] && sh->idx[r] && sh->particles[0][r] && sh->particles[1][r] &&
                         sh->llpr[0][r] && sh->llpr[1][r],
                     "bk_smc_shard: rank %d has a null buffer", r);
    return BK_OK;
}
static int shift_bits_for(int64_t M) {
    int lg = 0;
    while ((1ll << lg) < M) ++lg;
    return 61 - lg;
}

static int stat_blocks(int64_t M) {
    int64_t b = (M + RED_THREADS - 1) / RED_THREADS;
    return (int)(b < 1 ? 1 : (b > 1184 ? 1184 : b));  // 8 x 148 SMs
}

}  // namespace bk

using namespace bk;

extern "C" {

int bk_smc_move_weight(uint64_t handle, void* thetas, int64_t M, int32_t n, int32_t T, double scale,
                       const bk_rng* rng, void* logw_out, int32_t* accept_out, void* stream) {
    return bk_smc_gather_move_weight(handle, thetas, nullptr, thetas, M, n, T, scale, rng, logw_out,
                                     accept_out, stream);
}

int bk_smc_gather_move_weight(uint64_t handle, const void* src, const int64_t* src_idx, void* thetas,
                              int64_t M, int32_t n, int32_t T, double scale, const bk_rng* rng,
                              void* logw_out, int32_t* accept_out, void* stream) {
    return bk_smc_gather_move_weight_acc(handle, src, src_idx, thetas, M, n, T, scale, rng, nullptr, logw_out,
                                         accept_out, stream);
}

int bk_smc_gather_move_weight_acc(uint64_t handle, const void* src, const int64_t* src_idx, void* thetas,
                                  int64_t M, int32_t n, int32_t T, double scale, const bk_rng* rng,
                                  const void* logw_prev, void* logw_out, int32_t* accept_out, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    bk_smc_kernel kn = {BK_SMC_KERNEL_RW, 0, scale};
    if (int rc = check_smc_model(*m, kn)) return rc;
    BK_CHECK_ARG(src && thetas && logw_out && rng && M >= 0, "bk_smc_move_weight: bad argument");
    BK_CHECK_ARG(!src_idx || src != thetas,
                 "bk_smc_gather_move_weight: a gathered move cannot run in place (src == thetas)");
    BK_CHECK_ARG(T >= 1 && n >= 1 && n <= T, "bk_smc_move_weight: need 1 <= n <= T (n=%d, T=%d)", n, T);
    BK_CHECK_ARG(rng->mode != BK_RNG_INJECTED || (rng->normals && rng->uniforms && rng->n_uniform >= 1),
                 "bk_smc_move_weight: injected rng needs normals/uniforms");
    if (M == 0) return BK_OK;
    if (m->d.dtype == BK_F64)
        return smc_move_t<double>(*m, src, src_idx, thetas, M, n, T, kn, rng, logw_out, logw_prev, accept_out,
                                  (cudaStream_t)stream);
    return smc_move_t<float>(*m, src, src_idx, thetas, M, n, T, kn, rng, logw_out, logw_prev, accept_out,
                             (cudaStream_t)stream);
}

size_t bk_smc_resample_workspace_bytes(int64_t M) {
    if (M <= 0) return 256;
    size_t nb_scan = (size_t)((M + SCAN_TILE - 1) / SCAN_TILE);
    // max partials, sum partials, block totals + grand, cdf
    return align_up(1184 * 8, 256) + align_up(2 * 1184 * 8, 256) + align_up((nb_scan + 1) * 8, 256) +
           align_up((size_t)M * 8, 256) + 1024;
}

int bk_smc_weight_stats(const void* logw, int64_t M, int32_t dtype, int32_t mode, double* stats_out,
                        void* ws, size_t ws_bytes, void* stream) {
    BK_CHECK_ARG(logw && stats_out && M >= 1, "bk_smc_weight_stats: bad argument");
    Arena ar(ws, ws_bytes);
    double* maxp = ar.take<double>(1184);
    double* sump = ar.take<double>(2 * 1184);
    if (!ar.ok()) { set_error("bk_smc_weight_stats: workspace too small"); return BK_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int nb = stat_blocks(M);
    const int shift = mode == BK_RESAMPLE_SYSTEMATIC;
    if (dtype == BK_F64) k_max_partial<double><<<nb, RED_THREADS, 0, st>>>((const double*)logw, M, maxp);
    else k_max_partial<float><<<nb, RED_THREADS, 0, st>>>((const float*)logw, M, maxp);
    BK_LAUNCH_CHECK();
    k_max_final<<<1, 256, 0, st>>>(maxp, nb, shift, stats_out);
    BK_LAUNCH_CHECK();
    if (dtype == BK_F64) k_sum_partial<double><<<nb, RED_THREADS, 0, st>>>((const double*)logw, M, stats_out, sump);
    else k_sum_partial<float><<<nb, RED_THREADS, 0, st>>>((const float*)logw, M, stats_out, sump);
    BK_LAUNCH_CHECK();
    k_stats_final<<<1, 256, 0, st>>>(sump, nb, stats_out);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

static int resample_impl(const void* logw, int64_t M, int32_t dtype, int32_t mode, double shift, double total,
                         const double* stats, const void* uniforms, const bk_rng* rng, int64_t n_points,
                         int64_t point_offset, int64_t* idx_out, void* cdf_out, void* ws, size_t ws_bytes,
                         void* stream) {
    BK_CHECK_ARG(logw && idx_out && M >= 1, "bk_smc_resample_indices: bad argument");
    BK_CHECK_ARG(mode == BK_RESAMPLE_MULTINOMIAL || mode == BK_RESAMPLE_SYSTEMATIC,
                 "bk_smc_resample_indices: bad mode %d", mode);
    BK_CHECK_ARG(uniforms || rng, "bk_smc_resample_indices: need uniforms or rng");
    BK_CHECK_ARG(stats || total > 0, "bk_smc_resample_indices: total weight must be > 0 (got %g)", total);
    BK_CHECK_ARG(n_points >= 0 && point_offset >= 0 && point_offset + n_points <= M,
                 "bk_smc_resample_indices: point range [%lld, %lld) outside [0, %lld)",
                 (long long)point_offset, (long long)(point_offset + n_points), (long long)M);
    Arena ar(ws, ws_bytes);
    ar.take<double>(1184);
    ar.take<double>(2 * 1184);
    const int nb = (int)((M + SCAN_TILE - 1) / SCAN_TILE);
    double* btot = ar.take<double>(nb + 1);
    double* cdf = cdf_out ? (double*)cdf_out : ar.take<double>(M);
    if (!ar.ok()) { set_error("bk_smc_resample_indices: workspace too small"); return BK_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == BK_F64)
        k_scan_local<double><<<nb, SCAN_THREADS, 0, st>>>((const double*)logw, M, shift, total, stats, mode,
                                                           cdf, btot);
    else
        k_scan_local<float><<<nb, SCAN_THREADS, 0, st>>>((const float*)logw, M, shift, total, stats, mode, cdf,
                                                          btot);
    BK_LAUNCH_CHECK();
    k_scan_blocks<<<1, 1024, 0, st>>>(btot, nb, btot + nb);
    BK_LAUNCH_CHECK();
    k_scan_finish<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(cdf, M, btot, btot + nb);
    BK_LAUNCH_CHECK();
    bk_rng r;
    memset(&r, 0, sizeof(r));
    if (rng) r = *rng;
    if (n_points > 0) {
        const unsigned sb = (unsigned)((n_points + 255) / 256);
        if (dtype == BK_F64)
            k_search<double><<<sb, 256, 0, st>>>(cdf, M, mode, (const double*)uniforms, r, n_points,
                                                  point_offset, idx_out);
        else
            k_search<float><<<sb, 256, 0, st>>>(cdf, M, mode, (const float*)uniforms, r, n_points,
                                                 point_offset, idx_out);
        BK_LAUNCH_CHECK();
    }
    return BK_OK;
}

int bk_smc_resample_indices(const void* logw, int64_t M, int32_t dtype, int32_t mode, double shift,
                            double total, const void* uniforms, const bk_rng* rng, int64_t n_points,
                            int64_t point_offset, int64_t* idx_out, void* cdf_out, void* ws,
                            size_t ws_bytes, void* stream) {
    return resample_impl(logw, M, dtype, mode, shift, total, nullptr, uniforms, rng, n_points, point_offset,
                         idx_out, cdf_out, ws, ws_bytes, stream);
}

int bk_smc_resample_indices_dev(const void* logw, int64_t M, int32_t dtype, int32_t mode, const double* stats,
                                const void* uniforms, const bk_rng* rng, int64_t n_points,
                                int64_t point_offset, int64_t* idx_out, void* cdf_out, void* ws,
                                size_t ws_bytes, void* stream) {
    BK_CHECK_ARG(stats, "bk_smc_resample_indices_dev: stats is required");
    return resample_impl(logw, M, dtype, mode, 0.0, 1.0, stats, uniforms, rng, n_points, point_offset, idx_out,
                         cdf_out, ws, ws_bytes, stream);
}

int bk_smc_adaptive_select(const double* stats, double ess_threshold, int64_t n_points, int64_t point_offset,
                           int64_t* idx_inout, void* logw_inout, int32_t dtype, int32_t* resampled_out, void* stream) {
    BK_CHECK_ARG(stats && idx_inout && logw_inout && n_points >= 0, "bk_smc_adaptive_select: bad argument");
    const unsigned blocks = (unsigned)((n_points + 255) / 256 > 0 ? (n_points + 255) / 256 : 1);
    if (dtype == BK_F64)
        k_smc_adaptive_select<double><<<blocks, 256, 0, (cudaStream_t)stream>>>(stats, ess_threshold, n_points, point_offset,
                                                                               idx_inout, (double*)logw_inout, resampled_out);
    else
        k_smc_adaptive_select<float><<<blocks, 256, 0, (cudaStream_t)stream>>>(stats, ess_threshold, n_points, point_offset,
                                                                              idx_inout, (float*)logw_inout, resampled_out);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

int bk_gather_rows(const void* src, const int64_t* idx, int64_t M, int64_t D, int32_t dtype, void* out,
                   void* stream) {
    BK_CHECK_ARG(src && idx && out && M >= 0 && D >= 1, "bk_gather_rows: bad argument");
    if (M == 0) return BK_OK;
    const unsigned blocks = (unsigned)((M * 32 + 255) / 256);
    if (dtype == BK_F64)
        k_gather<double><<<blocks, 256, 0, (cudaStream_t)stream>>>((const double*)src, idx, M, (int)D, (double*)out);
    else
        k_gather<float><<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)src, idx, M, (int)D, (float*)out);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

// ---- sharded particle system -----------------------------------------------------------------
size_t bk_smc_shard_workspace_bytes(int64_t M, int32_t world, int32_t mode) {
    if (M < 1 || world < 1) return 256;
    size_t n = shard_ws_layout(nullptr, 0, M, world, nullptr) + 256;
    if (mode == BK_RESAMPLE_MULTINOMIAL) n += align_up((size_t)M * 8, 256) + bk_smc_resample_workspace_bytes(M) + 256;
    return n;
}

}  // extern "C"
template <typename T>
static int shard_move_t(const Model& m, const bk_smc_shard* sh, const ShardGeom& g, const void* src_local, int n, int Tn,
                        const bk_smc_kernel& kn, const bk_rng* rng, int accumulate, int32_t* accept, const ShardWs& w,
                        cudaStream_t st) {
    SmcArgs<T> a;
    memset(&a, 0, sizeof(a));
    const int cur = (int)(sh->epoch & 1), prev = cur ^ 1;
    a.thetas = (T*)sh->particles[cur][g.rank];
    a.M = shard_n(g, g.rank);
    a.sh = g;
    for (int r = 0; r < g.world; ++r) {
        a.src_tab[r] = (const T*)sh->particles[prev][r];
        a.llpr_tab[r] = (const T*)sh->llpr[prev][r];
        a.mail_tab[r] = (uint64_t*)sh->mailbox[r];
    }
    a.llpr_out = (T*)sh->llpr[cur][g.rank];
    a.carry = src_local ? 0 : 1;
    if (src_local) {
        a.src = (const T*)src_local;
        a.src_idx = nullptr;
    } else {
        a.src = (const T*)sh->particles[prev][g.rank];
        a.src_idx = sh->idx[g.rank];
    }
    // from the second step on, nothing of ours may be overwritten (log-weights, the older particle
    // array) before every rank has finished the previous step's reads: wait for their done messages
    a.wait_done = sh->epoch >= 2 ? sh->epoch - 1 : 0;
    a.epoch = sh->epoch;
    a.t0 = (T)((double)(n - 1) / Tn);  // smc.py:43-44
    a.t1 = (T)((double)n / Tn);
    a.rng = *rng;
    a.logw = (T*)sh->logw[g.rank];
    a.logw_prev = accumulate ? (const T*)sh->logw[g.rank] : nullptr;
    a.accept = accept;
    a.maxpart = w.maxpart;
    a.ticket = w.ctrl + CT_MOVE;
    return smc_dispatch<T>(m, a, kn, st);
}

extern "C" {
int bk_smc_shard_move(uint64_t handle, const bk_smc_shard* sh, const void* src_local, int32_t n, int32_t T,
                      const bk_smc_kernel* kernel, const bk_rng* rng, int32_t accumulate, int32_t* accept_out,
                      void* ws, size_t ws_bytes, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(kernel && rng, "bk_smc_shard_move: null argument");
    if (int rc = check_smc_model(*m, *kernel, rng)) return rc;
    ShardGeom g;
    if (int rc = make_geom(sh, &g)) return rc;
    BK_CHECK_ARG(T >= 1 && n >= 1 && n <= T, "bk_smc_shard_move: need 1 <= n <= T (n=%d, T=%d)", n, T);
    BK_CHECK_ARG(src_local || sh->epoch >= 2, "bk_smc_shard_move: the first step needs src_local");
    BK_CHECK_ARG(rng->mode != BK_RNG_INJECTED || (rng->normals && rng->uniforms && rng->n_uniform >= 1),
                 "bk_smc_shard_move: injected rng needs normals/uniforms");
    BK_CHECK_ARG(src_local != sh->particles[sh->epoch & 1][g.rank], "bk_smc_shard_move: src_local aliases the output array");
    ShardWs w;
    if (shard_ws_layout(ws, ws_bytes, sh->M, sh->world, &w) > ws_bytes || !ws) {
        set_error("bk_smc_shard_move: workspace too small");
        return BK_E_WORKSPACE;
    }
    if (m->d.dtype == BK_F64)
        return shard_move_t<double>(*m, sh, g, src_local, n, T, *kernel, rng, accumulate, accept_out, w, (cudaStream_t)stream);
    return shard_move_t<float>(*m, sh, g, src_local, n, T, *kernel, rng, accumulate, accept_out, w, (cudaStream_t)stream);
}

int bk_smc_shard_resample(const bk_smc_shard* sh, int32_t dtype, int32_t mode, const void* uniforms, const bk_rng* rng,
                          double ess_threshold, int32_t phase, double* stats_out, void* ws, size_t ws_bytes,
                          void* stream) {
    ShardGeom g;
    if (int rc = make_geom(sh, &g)) return rc;
    BK_CHECK_ARG(mode == BK_RESAMPLE_MULTINOMIAL || mode == BK_RESAMPLE_SYSTEMATIC, "bk_smc_shard_resample: bad mode %d", mode);
    BK_CHECK_ARG(uniforms || rng, "bk_smc_shard_resample: need uniforms or rng");
    BK_CHECK_ARG(phase >= 0 && phase <= 2, "bk_smc_shard_resample: phase must be 0, 1 or 2");
    BK_CHECK_ARG(!(ess_threshold > 0) || mode == BK_RESAMPLE_SYSTEMATIC,
                 "bk_smc_shard_resample: adaptive resampling needs the systematic mode");
    ShardWs w;
    if (shard_ws_layout(ws, ws_bytes, sh->M, sh->world, &w) > ws_bytes || !ws) {
        set_error("bk_smc_shard_resample: workspace too small");
        return BK_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = shard_n(g, g.rank);
    bk_rng r;
    memset(&r, 0, sizeof(r));
    if (rng) r = *rng;
    if (mode == BK_RESAMPLE_SYSTEMATIC) {
        const int s_bits = shift_bits_for(sh->M);
        if (phase == 0 || phase == 1) {
            ScanArgs a;
            memset(&a, 0, sizeof(a));
            a.logw = sh->logw[g.rank];
            a.n = n;
            a.shift_bits = s_bits;
            a.sh = g;
            for (int q = 0; q < g.world; ++q) a.mail_tab[q] = (uint64_t*)sh->mailbox[q];
            a.epoch = sh->epoch;
            a.cum = w.cum;
            a.tile_off = w.tile_off;
            a.qpart = w.qpart;
            a.ctrl = w.ctrl;
            a.n_tiles = (n + SC_TILE - 1) / SC_TILE;
            if (dtype == BK_F64) k_smc_scan<double><<<(unsigned)a.n_tiles, SC_THREADS, 0, st>>>(a);
            else k_smc_scan<float><<<(unsigned)a.n_tiles, SC_THREADS, 0, st>>>(a);
            BK_LAUNCH_CHECK();
        }
        if (phase == 0 || phase == 2) {
            ResolveArgs a;
            memset(&a, 0, sizeof(a));
            a.sh = g;
            for (int q = 0; q < g.world; ++q) {
                a.mail_tab[q] = (uint64_t*)sh->mailbox[q];
                a.idx_tab[q] = sh->idx[q];
            }
            a.epoch = sh->epoch;
            a.cum = w.cum;
            a.tile_off = w.tile_off;
            a.n = n;
            a.n_tiles = (n + SC_TILE - 1) / SC_TILE;
            a.shift_bits = s_bits;
            a.u0_in = uniforms;
            a.rng = r;
            a.ess_threshold = ess_threshold;
            a.logw = sh->logw[g.rank];
            a.stats_out = stats_out;
            a.ctrl = w.ctrl;
            // the expected number of points per rank is n; a rank holding most of the mass gets more (grid-stride)
            int64_t blocks = (n + 256 * RS_POINTS - 1) / (256 * RS_POINTS);
            const int64_t cap = (int64_t)device_sms() * 4;
            if (blocks > cap) blocks = cap;
            if (blocks < 1) blocks = 1;
            if (dtype == BK_F64) k_smc_resolve<double><<<(unsigned)blocks, 256, 0, st>>>(a);
            else k_smc_resolve<float><<<(unsigned)blocks, 256, 0, st>>>(a);
            BK_LAUNCH_CHECK();
        }
        return BK_OK;
    }
    // MULTINOMIAL (the reference's np.random.choice): full fp64 CDF on every rank
    if (phase == 2) return BK_OK;
    const size_t esz = dtype == BK_F64 ? 8 : 4;
    Arena ar(w.extra, w.extra_bytes);
    char* all = ar.take<char>((size_t)sh->M * 8);
    char* rws = ar.take<char>(0);
    const size_t rws_bytes = w.extra_bytes > ar.off ? w.extra_bytes - ar.off : 0;
    if (!ar.ok() || rws_bytes < bk_smc_resample_workspace_bytes(sh->M)) {
        set_error("bk_smc_shard_resample: workspace too small for the multinomial mode");
        return BK_E_WORKSPACE;
    }
    (void)esz;
    {
        CollectArgs a;
        memset(&a, 0, sizeof(a));
        a.sh = g;
        a.mailbox = (uint64_t*)sh->mailbox[g.rank];
        for (int q = 0; q < g.world; ++q) a.logw_tab[q] = sh->logw[q];
        a.epoch = sh->epoch;
        a.out = all;
        int64_t blocks = (sh->M + 255) / 256;
        if (blocks > 1184) blocks = 1184;
        if (dtype == BK_F64) k_smc_collect<double><<<(unsigned)blocks, 256, 0, st>>>(a);
        else k_smc_collect<float><<<(unsigned)blocks, 256, 0, st>>>(a);
        BK_LAUNCH_CHECK();
    }
    double* stats = stats_out ? stats_out : (double*)(w.maxpart);   // maxpart is idle between move kernels
    if (int rc = bk_smc_weight_stats(all, sh->M, dtype, mode, stats, rws, rws_bytes, stream)) return rc;
    if (int rc = resample_impl(all, sh->M, dtype, mode, 0.0, 1.0, stats, uniforms, rng, n, shard_lo(g, g.rank),
                               sh->idx[g.rank], nullptr, rws, rws_bytes, stream))
        return rc;
    DoneArgs d;
    memset(&d, 0, sizeof(d));
    d.sh = g;
    for (int q = 0; q < g.world; ++q) d.mail_tab[q] = (uint64_t*)sh->mailbox[q];
    d.epoch = sh->epoch;
    k_smc_post_done<<<1, 32, 0, st>>>(d);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

int bk_smc_shard_run(uint64_t handle, const bk_smc_shard* sh, const void* src_local, int32_t n_from, int32_t n_to,
                     int32_t T, const bk_smc_kernel* kernel, const bk_rng* rng, int32_t mode, double ess_threshold,
                     double* stats_out, int32_t* accept_out, void* ws, size_t ws_bytes, void* stream) {
    BK_CHECK_ARG(sh && rng && kernel, "bk_smc_shard_run: null argument");
    BK_CHECK_ARG(rng->mode == BK_RNG_PHILOX, "bk_smc_shard_run: device Philox only (injected streams go step by step)");
    BK_CHECK_ARG(n_from >= 1 && n_from <= n_to && n_to <= T, "bk_smc_shard_run: need 1 <= n_from <= n_to <= T");
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    bk_smc_shard s = *sh;
    for (int32_t n = n_from; n <= n_to; ++n) {
        bk_rng r = *rng;
        r.draw_offset = (uint64_t)n;
        const int accumulate = (ess_threshold > 0 && s.epoch > 1) ? 1 : 0;
        int rc = bk_smc_shard_move(handle, &s, n == n_from ? src_local : nullptr, n, T, kernel, &r, accumulate,
                                   n == n_to ? accept_out : nullptr, ws, ws_bytes, stream);
        if (rc) return rc;
        bk_rng rr = *rng;
        rr.draw_offset = (uint64_t)n;
        rr.chain_offset = 0;
        rc = bk_smc_shard_resample(&s, m->d.dtype, mode, nullptr, &rr, ess_threshold, 0,
                                   stats_out ? stats_out + 4 * (n - n_from) : nullptr, ws, ws_bytes, stream);
        if (rc) return rc;
        s.epoch += 1;
    }
    return BK_OK;
}

int bk_smc_cuda_prepare(uint64_t model, uint64_t proposal, char* log_out, size_t log_bytes) {
    if (log_out && log_bytes) log_out[0] = '\0';
    const Model* m = get_model(model);
    if (!m) return BK_E_HANDLE;
    const UserProposal* p = get_proposal(proposal);
    if (!p) return BK_E_HANDLE;
    bk_smc_kernel kn = {BK_SMC_KERNEL_PROPOSAL, 0, 0.0, proposal};
    if (int rc = check_smc_model(*m, kn)) return rc;
    return user_mhp_prepare(*m, *p, "bk_smc_cuda_prepare", log_out, log_bytes);
}

int bk_smc_shard_gather(const bk_smc_shard* sh, int64_t D, int32_t dtype, void* out, void* stream) {
    ShardGeom g;
    if (int rc = make_geom(sh, &g)) return rc;
    BK_CHECK_ARG(out && D >= 1, "bk_smc_shard_gather: bad argument");
    GatherArgs a;
    memset(&a, 0, sizeof(a));
    a.sh = g;
    a.mailbox = (uint64_t*)sh->mailbox[g.rank];
    for (int q = 0; q < g.world; ++q) a.src_tab[q] = sh->particles[sh->epoch & 1][q];
    a.idx = sh->idx[g.rank];
    a.epoch = sh->epoch;
    a.n = shard_n(g, g.rank);
    a.D = (int)D;
    a.out = out;
    int64_t blocks = (a.n * 32 + 255) / 256;
    const int64_t cap = (int64_t)device_sms() * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (dtype == BK_F64) k_smc_gather_sharded<double><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    else k_smc_gather_sharded<float><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

}  // extern "C"
