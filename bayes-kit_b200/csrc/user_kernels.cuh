// Kernels of user-written CUDA programs (BK_MODEL_USER_CUDA models and user proposals, bk.h).  The host side
// (user_model.cu, smc.cu) includes this file for the launch-argument structs and the program kinds only; the kernels
// are compiled at run time by NVRTC, one program per kind and key (user_model.cu), from
//   integer typedefs + device_rng.cuh + `typedef float|double bk_real;` [+ the model's source [+ smc_mailbox.cuh]]
//   [+ the proposal's source inside namespace bk_proposal] + this file
// with -DBK_DIMS=D and -DBK_PROGRAM=<kind>, which selects one of the sections at the end of this file:
//   BK_PROGRAM_MODEL            bk_user_eval; bk_user_hmc / mala / mh (D <= BK_USER_FUSED_MAX_D); prior/likelihood
//                               models also bk_user_eval_pl and bk_user_smc_rw / mala / hmc
//   BK_PROGRAM_PROPOSAL         bk_user_propose
//   BK_PROGRAM_MODEL_PROPOSAL   bk_user_mhp; prior/likelihood models also bk_user_smc_mhp
//   BK_PROGRAM_DRGHMC           bk_user_drghmc (also compiled with -DBK_DRGHMC=1, which the model's source may test)
//   BK_PROGRAM_STRETCH          bk_user_stretch (also compiled with -DBK_STRETCH=1, which the model's source may test)
// -DBK_SMC_KERNELS=1 marks the programs that carry SMC kernels (prior/likelihood models, kinds MODEL and
// MODEL_PROPOSAL): exactly those into which smc_mailbox.cuh is spliced.
// A model's source defines either
//   __device__ bk_real log_density_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
// or (bk_model_create_cuda_prior_lik: compiled with -DBK_PRIOR_LIK=1) the pair
//   __device__ bk_real log_prior_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
//   __device__ bk_real log_likelihood_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
// from which this file derives log_density_gradient = likelihood + prior.  A proposal's source defines propose() and,
// with -DBK_PROPOSAL_TRANSITION=1, transition_log_density() (bk.h), for -DBK_PROPOSAL_NORMALS / _UNIFORMS streams.
//
// bk_user_eval      one thread per chain on global rows: model_eval's case for this kind, through which the
//                   generic HMC / MALA / RW-Metropolis engine, the lockstep DrGHMC engine and the Stretcher's
//                   three-launch engine run.
// bk_user_hmc/mala/mh
//                   fused samplers, one thread per chain: theta, its gradient and log density stay in registers
//                   across all n_draws of a call.  Randomness and arithmetic follow the generic engine exactly
//                   (Row<T> and k_hmc_* / k_mala_* / k_mh_* in sampler_generic.cu): philox_normal4 per block of 4
//                   elements, philox_accept_uniform at block ceil(D / 4), the same sequence of Ar<T> operations;
//                   in fp64 only the summation order of the kinetic / proposal-energy sums differs.
// bk_user_eval_pl   (prior/likelihood models) log_prior and log_likelihood of global rows, one thread per row.
// bk_user_smc_rw/mala/hmc
//                   (prior/likelihood models) TemperedLikelihoodSMC's move + importance-weight kernel, one thread
//                   per particle: k_smc_move_weight (smc.cu) step for step with one lane per particle, on the same
//                   Philox words, the same resample-index / peer-row / (ll, prior)-carry rules and the same mailbox
//                   posts (smc_mailbox.cuh).
// bk_user_propose   one draw of a user proposal for global rows, one thread per chain: the propose step of the
//                   three-launch Metropolis(-Hastings) path.
// bk_user_mhp       Metropolis / MetropolisHastings with a user proposal fused with a user model, one thread per
//                   chain: bk_user_mh with propose() in place of the random walk.
// bk_user_smc_mhp   (prior/likelihood models) TemperedLikelihoodSMC's move + weight kernel with one
//                   Metropolis(-Hastings) step of the user's proposal as the move: bk_user_smc_rw with propose() in
//                   place of the random walk (BK_SMC_KERNEL_PROPOSAL).
// bk_user_drghmc    DrGhmcDiag, one thread per chain: k_drghmc (drghmc.cu) on the arithmetic and streams of the
//                   lockstep engine (drghmc_generic.cu).
// bk_user_stretch   one half-step of the Stretcher, one thread per active walker: k_stretch_propose, the density of
//                   the proposal and k_stretch_accept (ensemble.cu) in one launch, on the same uniforms and arithmetic.
#pragma once
#ifndef __CUDACC_RTC__
#include "smc_mailbox.cuh"
#endif

#define BK_PROGRAM_MODEL 1
#define BK_PROGRAM_PROPOSAL 2
#define BK_PROGRAM_MODEL_PROPOSAL 3
#define BK_PROGRAM_DRGHMC 4
#define BK_PROGRAM_STRETCH 5

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
    const void* prop_params;  // bk_user_mhp: the proposal's [n_params] or NULL
};

#if !defined(__CUDACC_RTC__) || BK_PROGRAM == BK_PROGRAM_DRGHMC
// Launch arguments of bk_user_drghmc.  `run` holds what bk_user_hmc reads (theta, params, metric, the streams with
// n_uniform = 2K when injected, draws / logp / accept); step sizes and the damping terms are rounded to the dtype in
// the kernel, as the lockstep engine rounds them on the host.
constexpr int USER_DR_KMAX = 6;   // drghmc.cu's DR_KMAX: bk_drghmc_sample refuses a larger K before dispatching
struct UserDrArgs {
    UserRunArgs run;
    void* rho;                        // [C, D] in/out: the persistent momentum
    int32_t* n_used;                  // [n, C] uniforms consumed per draw, or NULL
    int32_t K, prob_retry;
    int32_t cnt[USER_DR_KMAX];        // leapfrog steps of proposal k
    double eps[USER_DR_KMAX], half_eps[USER_DR_KMAX];
    double s_keep, s_new;             // sqrt(1 - damping), sqrt(damping)
};
#endif

#if !defined(__CUDACC_RTC__) || BK_PROGRAM == BK_PROGRAM_STRETCH
// Launch arguments of bk_user_stretch: one half-step of the Stretcher (bk_stretch_move).  lo / width are rounded to
// the dtype in the kernel, as stretch_t (ensemble.cu) rounds them on the host.
struct UserStretchArgs {
    void* active;             // [n, D] in/out: the walkers that move
    void* lp;                 // [n] in/out: their cached log densities
    const void* other;        // [m, D] the complementary walkers
    int32_t* accept;          // [n] or NULL
    const void* params;       // [n_params] or NULL
    const void* uniforms;     // injected [n, 3]: partner, stretch, accept
    int64_t n, m;
    double lo, width;         // u_z = lo + width * u1: 1 / sqrt(a), sqrt(a) - 1 / sqrt(a)
    uint64_t seed, draw_offset, chain_offset;
    int32_t rng_mode, n_uniform;   // n_uniform = 3
    int32_t eval_lp;          // evaluate log p(active) first (the cache is invalid) and store it
};
#endif

// Launch arguments of bk_user_propose (one draw of a user proposal for C chains, three-launch path).  Streams: injected
// normals [n, C, BK_PROPOSAL_NORMALS] and uniforms [n, C, n_uniform] (column 0: the accept uniform, columns 1 + k:
// u[k]); in Philox mode the kernel writes this draw's z / u into zbuf [C, BK_PROPOSAL_NORMALS] / ubuf
// [C, BK_PROPOSAL_UNIFORMS] and hands the proposal those rows.
struct UserProposeArgs {
    const void* theta;        // [C, D]
    void* q;                  // [C, D] out
    void* dh;                 // [C] out: log q(theta | q) - log q(q | theta), or NULL (no Hastings term)
    const void* params;       // [n_params] or NULL
    const void* normals;
    const void* uniforms;
    void* zbuf;
    void* ubuf;
    int64_t C, t;             // t: draw of this call
    uint64_t seed, draw_offset, chain_offset;
    int32_t rng_mode, n_uniform;
};

#if !defined(__CUDACC_RTC__) || defined(BK_SMC_KERNELS)
// Launch arguments of bk_user_smc_rw / _mala / _hmc / _mhp: SmcArgs<T> of smc.cu with plain fields (the host (nvcc) and
// the kernels (NVRTC) must agree on the layout).  Pointers are in the model's dtype unless typed.
struct UserSmcArgs {
    void* thetas;                          // [M, D] moved particles (out)
    const void* src;                       // particles to move: row src_idx[m] (the pending resample) or row m
    const int64_t* src_idx;                // [M] or NULL
    int64_t M;
    double t0, t1;                         // temperatures, already rounded to the dtype
    double scale;                          // RW: proposal sd; MALA: epsilon; HMC: stepsize
    int32_t steps;                         // HMC: leapfrog steps
    int32_t rng_mode, n_uniform;           // bk_rng
    uint64_t seed, draw_offset, chain_offset;
    const void* normals;                   // injected [M, D]
    const void* uniforms;                  // injected [M, n_uniform]
    void* logw;                            // [M] out
    const void* logw_prev;                 // [M] carried log-weights or NULL
    int32_t* accept;                       // [M] or NULL
    // ---- sharded particle system (smc_mailbox.cuh); sh.world == 0: plain single-array call ----
    ShardGeom sh;                          // src_idx holds GLOBAL particle ids, row gid lives on rank owner(gid)
    const void* src_tab[BK_SMC_MAX_WORLD];
    const void* llpr_tab[BK_SMC_MAX_WORLD];
    uint64_t* mail_tab[BK_SMC_MAX_WORLD];
    void* llpr_out;                        // [M, 2] (log_likelihood, log_prior) of the moved particles, or NULL
    int32_t carry;                         // read the parent's pair from llpr_tab instead of evaluating the model
    uint64_t epoch, wait_done;
    double* maxpart;                       // [gridDim.x] per-CTA maxima (NULL: no statistics epilogue)
    unsigned* ticket;
    const void* params;                    // [n_params] or NULL
    const void* prop_params;               // bk_user_smc_mhp: the proposal's [n_params] or NULL
};
#endif

}  // namespace bk

#ifdef __CUDACC_RTC__

#ifdef BK_PRIOR_LIK
// The posterior's density from the pair, in the order of the built-in GAUSS_PRIOR_LIK evaluator (k_sep_eval):
// lp = ll + prior, grad = gll + gpr.
__device__ __forceinline__ bk_real log_density_gradient(const bk_real* theta, bk_real* grad, const bk_real* params) {
    using A = bk::Ar<bk_real>;
    bk_real gpr[BK_DIMS];
    const bk_real pr = log_prior_gradient(theta, gpr, params);
    const bk_real ll = log_likelihood_gradient(theta, grad, params);
#pragma unroll
    for (int e = 0; e < BK_DIMS; ++e) grad[e] = A::add(grad[e], gpr[e]);
    return A::add(ll, pr);
}
#endif

namespace bk {
namespace user {

constexpr int D = BK_DIMS;
constexpr int NB = (D + 3) / 4;   // element blocks of 4
using T = bk_real;
using A = Ar<T>;

// ---- the random streams ---------------------------------------------------------------------------------------------
// S is a launch-argument struct (its bk_rng fields).  A launch reads draw t of chain c: injected streams are
// [n, C, width] arrays read at row t * C + c, Philox words are keyed by the global chain chain_offset + c and the
// global draw draw_offset + t.  The SMC's move is one draw (t = 0) of C = M particles.  C is taken by reference so
// that it is loaded, and the row formed, in the injected branch only: passed by value, its load moves ahead of the
// branch and ptxas schedules the fused samplers differently.
template <class S>
__device__ __forceinline__ uint32_t chain_word(const S& s, int64_t c) {
    return (uint32_t)(s.chain_offset + (uint64_t)c);
}
template <class S>
__device__ __forceinline__ uint32_t draw_word(const S& s, int64_t t) {
    return (uint32_t)(s.draw_offset + (uint64_t)t);
}

// normals of element block b: the rule of Row<T>::normal4
template <class S>
__device__ __forceinline__ void normal4(const S& s, const int64_t& C, int64_t c, int64_t t, int b, T (&z)[4]) {
    if (s.rng_mode == 1) {   // BK_RNG_INJECTED
        const T* p = reinterpret_cast<const T*>(s.normals) + (t * C + c) * (int64_t)D;
#pragma unroll
        for (int i = 0; i < 4; ++i) z[i] = (4 * b + i < D) ? p[4 * b + i] : T(0);
    } else {
        philox_normal4<T>(s.seed, (uint32_t)b, chain_word(s, c), draw_word(s, t), z);
    }
}

// all D normals
template <class S>
__device__ __forceinline__ void normals(const S& s, const int64_t& C, int64_t c, int64_t t, T (&z)[D]) {
#pragma unroll
    for (int b = 0; b < NB; ++b) {
        T z4[4];
        normal4(s, C, c, t, b, z4);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (4 * b + i < D) z[4 * b + i] = z4[i];
    }
}

// the accept uniform: column 0 of the injected row, else the Philox accept block or, with `streams` (Row<T>::uniform(0)
// of a draw of several uniforms), TAG_UNIFORM word 0
template <class S>
__device__ __forceinline__ T accept_uniform(const S& s, const int64_t& C, int64_t c, int64_t t, bool streams = false) {
    if (s.rng_mode == 1) return reinterpret_cast<const T*>(s.uniforms)[(t * C + c) * s.n_uniform];
    if (!streams) return philox_accept_uniform<T>(s.seed, chain_word(s, c), draw_word(s, t), D);
    return philox_uniform<T>(s.seed, 0u, chain_word(s, c), draw_word(s, t));
}

// the k-th uniform: column k of the injected row, else TAG_UNIFORM word k (drg_uniform, drghmc_generic.cu)
template <class S>
__device__ __forceinline__ T uniform(const S& s, const int64_t& C, int64_t c, int64_t t, int k) {
    if (s.rng_mode == 1) return reinterpret_cast<const T*>(s.uniforms)[(t * C + c) * s.n_uniform + k];
    return philox_uniform<T>(s.seed, (uint32_t)k, chain_word(s, c), draw_word(s, t));
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

// ---- what a proposal's programs share -------------------------------------------------------------------------------
#if BK_PROGRAM == BK_PROGRAM_PROPOSAL || BK_PROGRAM == BK_PROGRAM_MODEL_PROPOSAL

namespace bk {
namespace user {

constexpr int NZ = BK_PROPOSAL_NORMALS, NU = BK_PROPOSAL_UNIFORMS;
constexpr int NZ1 = NZ > 0 ? NZ : 1, NU1 = NU > 0 ? NU : 1;   // array extents

// the proposal's injected rows: normals [row, NZ]; uniforms [row, n_uniform], whose column 0 is the accept uniform
template <class S>
__device__ __forceinline__ const T* proposal_z(const S& s, int64_t row) {
    return reinterpret_cast<const T*>(s.normals) + row * NZ;
}
template <class S>
__device__ __forceinline__ const T* proposal_u(const S& s, int64_t row) {
    return reinterpret_cast<const T*>(s.uniforms) + row * s.n_uniform + 1;
}

// the proposal's Philox streams of (global chain, draw): z[k] from block proposal_normal_block(k, D), u[k] the k-th
// TAG_UNIFORM uniform
__device__ __forceinline__ void proposal_philox(uint64_t seed, uint32_t chain, uint32_t draw, T* z, T* u) {
#pragma unroll
    for (int b = 0; 4 * b < NZ; ++b) {
        T z4[4];
        philox_normal4<T>(seed, (uint32_t)proposal_normal_block(4 * b, D), chain, draw, z4);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (4 * b + i < NZ) z[4 * b + i] = z4[i];
    }
#pragma unroll
    for (int k = 0; k < NU; ++k) u[k] = philox_uniform<T>(seed, (uint32_t)k, chain, draw);
}

// the proposal's z / u into local arrays: copied from the injected rows or drawn from Philox
template <class S>
__device__ __forceinline__ void proposal_streams(const S& s, const int64_t& C, int64_t c, int64_t t, T (&z)[NZ1],
                                                 T (&u)[NU1]) {
    if (s.rng_mode == 1) {   // BK_RNG_INJECTED
        const int64_t r = t * C + c;
        const T* zi = proposal_z(s, r);
        const T* ui = proposal_u(s, r);
#pragma unroll
        for (int k = 0; k < NZ; ++k) z[k] = zi[k];
#pragma unroll
        for (int k = 0; k < NU; ++k) u[k] = ui[k];
    } else {
        proposal_philox(s.seed, chain_word(s, c), draw_word(s, t), z, u);
    }
}

// log q(theta | q) - log q(q | theta), in MetropolisHastings's order: fwd = q(proposal | theta), rev = q(theta | proposal)
__device__ __forceinline__ T proposal_dh(const T* th, const T* q, const T* pp) {
#if BK_PROPOSAL_TRANSITION
    const T fwd = bk_proposal::transition_log_density(q, th, pp);
    const T rev = bk_proposal::transition_log_density(th, q, pp);
    return A::sub(rev, fwd);
#else
    return T(0);
#endif
}

}  // namespace user
}  // namespace bk

#endif  // proposal programs

// ---- what the SMC kernels share -------------------------------------------------------------------------------------
#ifdef BK_SMC_KERNELS

namespace bk {
namespace user {

// (ll, prior) of x and the gradient of the tempered density lp_t = ll * t + prior: g = gll * t + gpr (smc.cu's tgrad)
__device__ __forceinline__ void tempered(const T (&x)[D], T t, const T* params, T& ll, T& pr, T (&g)[D]) {
    T gp[D];
    pr = log_prior_gradient(x, gp, params);
    ll = log_likelihood_gradient(x, g, params);
#pragma unroll
    for (int e = 0; e < D; ++e) g[e] = A::add(A::mul(g[e], t), gp[e]);
}

// k_smc_move_weight with one lane per particle.  MOVE: BK_SMC_KERNEL_RW / _MALA / _HMC / _PROPOSAL (bk.h: 0 .. 3).
template <int MOVE>
__device__ __forceinline__ void smc_move(const UserSmcArgs& a) {
    const T* params = reinterpret_cast<const T*>(a.params);
    const T t0 = (T)a.t0, t1 = (T)a.t1;
    const bool carry = a.carry != 0;
    // sharded source: the resample indices are global particle ids; the row is read from its owner's array
    const bool sharded = a.sh.world > 1 && a.src_idx != nullptr;
    if (a.wait_done) {   // the indices (and the rows they point at) of the previous step are final on every rank
        if ((int)threadIdx.x < a.sh.world)
            mail_wait(a.mail_tab[a.sh.rank] + MB_DONE + (a.wait_done & 1) * BK_SMC_MAX_WORLD + threadIdx.x, a.wait_done,
                      a.mail_tab[a.sh.rank]);
        __syncthreads();
    }
    double lw_max = (double)neg_inf<float>();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; m < a.M; m += stride) {
        const int64_t gid = a.src_idx ? a.src_idx[m] : m;
        const T* row;
        const T* llpr;
        if (sharded) {
            int r;
            int64_t loc;
            shard_locate(a.sh, gid, r, loc);
            row = reinterpret_cast<const T*>(a.src_tab[r]) + loc * (int64_t)D;
            llpr = reinterpret_cast<const T*>(a.llpr_tab[r]) + 2 * loc;
        } else {
            row = reinterpret_cast<const T*>(a.src) + gid * (int64_t)D;
            llpr = reinterpret_cast<const T*>(a.llpr_tab[a.sh.world > 0 ? a.sh.rank : 0]) + 2 * gid;
        }
        T th[D], st[D], z[D];
        load_row(row, th);
        // proposal normals: the words Lanes<T, G, J>::normals consumes for blocks 0 .. ceil(D / 4) - 1 (the user's
        // proposal draws its own streams below).  The loop is normals()'s, spelled out: through normals() ptxas
        // allocates the fp64 RW kernel's registers differently.
#pragma unroll
        for (int b = 0; b < (MOVE == 3 ? 0 : NB); ++b) {
            T z4[4];
            normal4(a, a.M, m, 0, b, z4);
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (4 * b + i < D) z[4 * b + i] = z4[i];
        }
        const T lu = log_u(accept_uniform(a, a.M, m, 0));
        T ll_c, pr_c, ll_s, pr_s;
        if (carry) { ll_c = llpr[0]; pr_c = llpr[1]; }
        bool acc;
        if constexpr (MOVE == 0) {   // RW (smc.py:79-89); the gradients are dead code after inlining
            T unused[D];
            if (!carry) tempered(th, t0, params, ll_c, pr_c, unused);
            const T lp_c = A::add(A::mul(ll_c, t0), pr_c);
#pragma unroll
            for (int e = 0; e < D; ++e) st[e] = A::add(th[e], A::mul((T)a.scale, z[e]));   // smc.py:81
            tempered(st, t0, params, ll_s, pr_s, unused);
            const T lp_s = A::add(A::mul(ll_s, t0), pr_s);
            acc = lu < A::sub(lp_s, lp_c);   // smc.py:85
        } else if constexpr (MOVE == 1) {   // one MALA transition on the tempered density (mala.py:40-66)
            const T eps = (T)a.scale, sd = A::sqrt_(A::mul(T(2), eps)), coef = T(-0.25) / eps;
            T g[D], gs[D], ll_e, pr_e;
            tempered(th, t0, params, ll_e, pr_e, g);
            if (!carry) { ll_c = ll_e; pr_c = pr_e; }
            const T lp_c = A::add(A::mul(ll_c, t0), pr_c);
#pragma unroll
            for (int e = 0; e < D; ++e) st[e] = A::add(A::add(th[e], A::mul(eps, g[e])), A::mul(sd, z[e]));
            tempered(st, t0, params, ll_s, pr_s, gs);
            const T lp_s = A::add(A::mul(ll_s, t0), pr_s);
            T sf = T(0), sr = T(0);
#pragma unroll
            for (int e = 0; e < D; ++e) {
                const T df = A::sub(A::sub(st[e], th[e]), A::mul(eps, g[e]));
                const T dr = A::sub(A::sub(th[e], st[e]), A::mul(eps, gs[e]));
                sf = A::add(sf, A::mul(df, df));
                sr = A::add(sr, A::mul(dr, dr));
            }
            const T fwd = A::mul(coef, sf), rev = A::mul(coef, sr);
            acc = lu < A::add(A::sub(lp_s, lp_c), A::sub(rev, fwd));   // metropolis.py:41-76
#if BK_PROGRAM == BK_PROGRAM_MODEL_PROPOSAL
        } else if constexpr (MOVE == 3) {   // the RW branch with the user's proposal: bk_user_mhp's step
            const T* pp = reinterpret_cast<const T*>(a.prop_params);
            T zp[NZ1], up[NU1], unused[D];
            proposal_streams(a, a.M, m, 0, zp, up);   // injected: normals [M, NZ], uniforms [M, 1 + NU]
            if (!carry) tempered(th, t0, params, ll_c, pr_c, unused);
            const T lp_c = A::add(A::mul(ll_c, t0), pr_c);
            bk_proposal::propose(th, st, zp, up, pp);
            tempered(st, t0, params, ll_s, pr_s, unused);
            const T lp_s = A::add(A::mul(ll_s, t0), pr_s);
            T ratio = A::sub(lp_s, lp_c);
#if BK_PROPOSAL_TRANSITION
            ratio = A::add(ratio, proposal_dh(th, st, pp));
#endif
            acc = lu < ratio;
#endif
        } else {   // one HMCDiag transition, identity metric, on the tempered density (hmc.py:40-63)
            const T eps = (T)a.scale, heps = A::mul(T(0.5), eps);
            T g[D];
            tempered(th, t0, params, ll_s, pr_s, g);   // (ll_s, pr_s): the terms at st, which starts at th
            if (!carry) { ll_c = ll_s; pr_c = pr_s; }
            const T lp_c = A::add(A::mul(ll_c, t0), pr_c);
            T kin = T(0);
#pragma unroll
            for (int e = 0; e < D; ++e) kin = A::add(kin, A::mul(z[e], z[e]));
            const T h0 = A::sub(lp_c, A::mul(T(0.5), kin));
#pragma unroll
            for (int e = 0; e < D; ++e) {   // backward half kick (hmc.py:46)
                st[e] = th[e];
                z[e] = A::sub(z[e], A::mul(heps, g[e]));
            }
            for (int s = 0; s < a.steps; ++s) {   // hmc.py:47-50
#pragma unroll
                for (int e = 0; e < D; ++e) {
                    z[e] = A::add(z[e], A::mul(eps, g[e]));
                    st[e] = A::add(st[e], A::mul(eps, z[e]));
                }
                tempered(st, t0, params, ll_s, pr_s, g);
            }
            kin = T(0);
#pragma unroll
            for (int e = 0; e < D; ++e) {   // forward half kick (hmc.py:52)
                z[e] = A::add(z[e], A::mul(heps, g[e]));
                kin = A::add(kin, A::mul(z[e], z[e]));
            }
            const T h1 = A::sub(A::add(A::mul(ll_s, t0), pr_s), A::mul(T(0.5), kin));
            acc = lu < A::sub(h1, h0);   // hmc.py:60
        }
        if (acc) {
#pragma unroll
            for (int e = 0; e < D; ++e) th[e] = st[e];
            ll_c = ll_s;
            pr_c = pr_s;
        }
        // importance log-weight, both tempered densities in full (smc.py:67-70)
        const T lw = A::sub(A::add(A::mul(ll_c, t1), pr_c), A::add(A::mul(ll_c, t0), pr_c));
        T* out = reinterpret_cast<T*>(a.thetas) + m * (int64_t)D;
#pragma unroll
        for (int e = 0; e < D; ++e) out[e] = th[e];
        if (a.llpr_out) {
            T* lo = reinterpret_cast<T*>(a.llpr_out) + 2 * m;
            lo[0] = ll_c;
            lo[1] = pr_c;
        }
        const T lw_tot = a.logw_prev ? A::add(reinterpret_cast<const T*>(a.logw_prev)[m], lw) : lw;
        reinterpret_cast<T*>(a.logw)[m] = lw_tot;
        lw_max = fmax(lw_max, (double)lw_tot);
        if (a.accept) a.accept[m] = acc ? 1 : 0;
    }
    if (a.maxpart) smc_post_max(lw_max, a.maxpart, a.ticket, a.sh, a.mail_tab, a.epoch);
}

}  // namespace user
}  // namespace bk

#endif  // BK_SMC_KERNELS

// =====================================================================================================================
// ---- BK_PROGRAM_MODEL: a model's own program (bk_model_create_cuda / _prior_lik) -----------------------------------
#if BK_PROGRAM == BK_PROGRAM_MODEL

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
        normals(a, a.C, c, t, r);
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
        const bool acc = bk::log_u(accept_uniform(a, a.C, c, t, a.n_uniform != 1)) < A::sub(h1, h0);
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
        normals(a, a.C, c, t, q);
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
        const bool acc = bk::log_u(accept_uniform(a, a.C, c, t, a.n_uniform != 1)) < A::add(A::sub(lpq, lp), A::sub(rev, fwd));
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
        normals(a, a.C, c, t, q);
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
        const bool acc = bk::log_u(accept_uniform(a, a.C, c, t, a.n_uniform != 1)) < ratio;
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

#ifdef BK_SMC_KERNELS

// theta [C, D] -> log_prior [C], log_likelihood [C] (each nullable)
extern "C" __global__ void __launch_bounds__(128) bk_user_eval_pl(const bk_real* __restrict__ theta, long long C,
                                                                  const bk_real* __restrict__ params,
                                                                  bk_real* __restrict__ lprior,
                                                                  bk_real* __restrict__ llik) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    bk_real g[BK_DIMS];
    const bk_real* x = theta + c * BK_DIMS;
    if (lprior) lprior[c] = log_prior_gradient(x, g, params);
    if (llik) llik[c] = log_likelihood_gradient(x, g, params);
}

extern "C" __global__ void __launch_bounds__(128) bk_user_smc_rw(const bk::UserSmcArgs a) { bk::user::smc_move<0>(a); }
extern "C" __global__ void __launch_bounds__(128) bk_user_smc_mala(const bk::UserSmcArgs a) { bk::user::smc_move<1>(a); }
extern "C" __global__ void __launch_bounds__(128) bk_user_smc_hmc(const bk::UserSmcArgs a) { bk::user::smc_move<2>(a); }

#endif  // BK_SMC_KERNELS

// ---- BK_PROGRAM_PROPOSAL: a proposal's own program (bk_proposal_create_cuda) ----------------------------------------
#elif BK_PROGRAM == BK_PROGRAM_PROPOSAL

// One draw of the proposal for every chain: q = propose(theta, z, u) and, when dh is given, the Hastings term.
extern "C" __global__ void __launch_bounds__(128) bk_user_propose(const bk::UserProposeArgs a) {
    using namespace bk::user;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.C) return;
    const T* pp = reinterpret_cast<const T*>(a.params);
    const T* th = reinterpret_cast<const T*>(a.theta) + c * (int64_t)D;
    T* q = reinterpret_cast<T*>(a.q) + c * (int64_t)D;
    const T *z, *u;
    if (a.rng_mode == 1) {   // BK_RNG_INJECTED: the proposal reads the rows in place
        const int64_t r = a.t * a.C + c;
        z = proposal_z(a, r);
        u = proposal_u(a, r);
    } else {   // Philox: through the scratch rows, so that a proposal of any size runs
        T* zw = reinterpret_cast<T*>(a.zbuf) + c * NZ;
        T* uw = reinterpret_cast<T*>(a.ubuf) + c * NU;
        proposal_philox(a.seed, chain_word(a, c), draw_word(a, a.t), zw, uw);
        z = zw;
        u = uw;
    }
    bk_proposal::propose(th, q, z, u, pp);
    if (a.dh) reinterpret_cast<T*>(a.dh)[c] = proposal_dh(th, q, pp);
}

// ---- BK_PROGRAM_MODEL_PROPOSAL: a model's and a proposal's sources in one program, compiled on first use -----------
#elif BK_PROGRAM == BK_PROGRAM_MODEL_PROPOSAL

// (defined first: ptxas then reports the two kernels in the order it always has)
#ifdef BK_SMC_KERNELS
extern "C" __global__ void __launch_bounds__(128) bk_user_smc_mhp(const bk::UserSmcArgs a) { bk::user::smc_move<3>(a); }
#endif

// Metropolis / MetropolisHastings with a user proposal, fused with the user's model: bk_user_mh with the random walk
// replaced by propose() and its Gaussian Hastings sum by transition_log_density.  The model's gradient is dead code.
extern "C" __global__ void __launch_bounds__(128) bk_user_mhp(const bk::UserRunArgs a) {
    using namespace bk::user;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.C) return;
    const T* params = reinterpret_cast<const T*>(a.params);
    const T* pp = reinterpret_cast<const T*>(a.prop_params);
    T* row = reinterpret_cast<T*>(a.theta) + c * (int64_t)D;
    T th[D], unused[D];
    load_row(row, th);
    T lp = log_density_gradient(th, unused, params);
    for (int64_t t = 0; t < a.n_draws; ++t) {
        T q[D], z[NZ1], u[NU1];
        proposal_streams(a, a.C, c, t, z, u);
        bk_proposal::propose(th, q, z, u, pp);
        const T lpq = log_density_gradient(q, unused, params);
        T ratio = A::sub(lpq, lp);
        if (a.hastings) ratio = A::add(ratio, proposal_dh(th, q, pp));
        const bool acc = bk::log_u(accept_uniform(a, a.C, c, t, a.n_uniform != 1)) < ratio;
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

// ---- BK_PROGRAM_DRGHMC: DrGhmcDiag on a model, compiled on first use ------------------------------------------------
// One chain per thread follows its own retry / accept / ghost schedule (drghmc.py:348-446) and integrates only the
// trajectories that schedule reaches; the lockstep engine integrates every trajectory a chain could need.  Every point
// carries its own (log p, grad log p), as the lockstep engine's levels do: theta's pair across attempts and draws, a
// proposal's from the last evaluation of its trajectory, so a trajectory of cnt steps costs cnt evaluations.
// The proposal recursion is compile-time (DrAccept<k>, the shape of drghmc.cu's Accept<k>) with a __noinline__ run()
// per level, and every trajectory goes through one __noinline__ trajectory(): the user's function is inlined twice
// (at entry and in trajectory()) whatever K is, which bounds NVRTC's work for a heavy model.
#elif BK_PROGRAM == BK_PROGRAM_DRGHMC

namespace bk {
namespace user {

struct DrCtx {
    const T* params;
    const T* metric;   // [D] or NULL (identity)
    T eps[USER_DR_KMAX], half[USER_DR_KMAX];
    int cnt[USER_DR_KMAX];
    int prob_retry;
};

// drghmc.py:317: bool * float (False * -inf = nan on purpose)
__device__ __forceinline__ T dr_retry(const DrCtx& c, T reject_logp) {
    return c.prob_retry ? reject_logp : A::mul(T(0), reject_logp);
}
__device__ __forceinline__ T dr_log1m_exp(T a) { return A::log1p_(-A::exp_(a)); }   // np.log1p(-np.exp(a))
__device__ __forceinline__ T dr_mg(const DrCtx& c, int e, T g) { return c.metric ? A::mul(c.metric[e], g) : g; }

// proposal_map (drghmc.py:319-346) of proposal i from (q0, r0, g0): k_drg_first, then cnt - 1 times (evaluate,
// k_drg_step), evaluate, k_drg_last.  Leaves the end point's pair in (lp, g) and returns its joint log density
// lp - kinetic(r).
__device__ __noinline__ T trajectory(const DrCtx& c, int i, const T (&q0)[D], const T (&r0)[D], const T (&g0)[D],
                                     T (&q)[D], T (&r)[D], T (&g)[D], T& lp) {
    const T eps = c.eps[i], half = c.half[i];
    T qq[D], rr[D], gg[D];
#pragma unroll
    for (int e = 0; e < D; ++e) {
        rr[e] = A::add(r0[e], A::mul(half, dr_mg(c, e, g0[e])));
        qq[e] = A::add(q0[e], A::mul(eps, rr[e]));
    }
    T l;
    for (int s = 1;; ++s) {
        l = log_density_gradient(qq, gg, c.params);
        if (s == c.cnt[i]) break;
#pragma unroll
        for (int e = 0; e < D; ++e) {
            rr[e] = A::add(rr[e], A::mul(eps, dr_mg(c, e, gg[e])));
            qq[e] = A::add(qq[e], A::mul(eps, rr[e]));
        }
    }
    T kin = T(0);
#pragma unroll
    for (int e = 0; e < D; ++e) {
        const T re = -A::add(rr[e], A::mul(half, dr_mg(c, e, gg[e])));
        kin = A::add(kin, A::mul(re, dr_mg(c, e, re)));
        q[e] = qq[e];
        r[e] = re;
        g[e] = gg[e];
    }
    lp = l;
    return A::sub(l, A::mul(T(0.5), kin));
}

// log acceptance probability of proposal K, the point (qp, rp, gp) with joint log density prop_logp, made from a state
// with (cur_hastings, cur_logp): drghmc.py:391-446
template <int K>
struct DrAccept {
    // ghosts I .. K - 1 of the point (drghmc.py:424-436); true on the early exit at accept_logp == 0
    template <int I>
    static __device__ __forceinline__ bool ghosts(const DrCtx& c, const T (&qp)[D], const T (&rp)[D],
                                                  const T (&gp)[D], T prop_logp, T& prop_hastings) {
        if constexpr (I < K) {
            T qg[D], rg[D], gg[D], lg;
            const T jg = trajectory(c, I, qp, rp, gp, qg, rg, gg, lg);
            const T ai = DrAccept<I>::run(c, qg, rg, gg, jg, prop_hastings, prop_logp);
            if (ai == T(0)) return true;
            prop_hastings = A::add(prop_hastings, dr_log1m_exp(ai));
            return ghosts<I + 1>(c, qp, rp, gp, prop_logp, prop_hastings);
        } else {
            return false;
        }
    }

    static __device__ __noinline__ T run(const DrCtx& c, const T (&qp)[D], const T (&rp)[D], const T (&gp)[D],
                                         T prop_logp, T cur_hastings, T cur_logp) {
        T prop_hastings = T(0);
        if (ghosts<0>(c, qp, rp, gp, prop_logp, prop_hastings)) return neg_inf<T>();
        const T frac = A::add(A::add(A::sub(prop_logp, cur_logp), A::sub(prop_hastings, cur_hastings)),
                              A::sub(dr_retry(c, prop_hastings), dr_retry(c, cur_hastings)));
        return frac < T(0) ? frac : T(0);   // python min(0, frac): nan -> 0
    }
};

// DrAccept<k>::run for a run-time k < K <= USER_DR_KMAX
template <int K>
__device__ __forceinline__ T dr_accept(int k, const DrCtx& c, const T (&qp)[D], const T (&rp)[D], const T (&gp)[D],
                                       T prop_logp, T cur_hastings, T cur_logp) {
    if constexpr (K < USER_DR_KMAX) {
        if (k == K) return DrAccept<K>::run(c, qp, rp, gp, prop_logp, cur_hastings, cur_logp);
        return dr_accept<K + 1>(k, c, qp, rp, gp, prop_logp, cur_hastings, cur_logp);
    } else {
        return neg_inf<T>();
    }
}

}  // namespace user
}  // namespace bk

// theta, rho [C, D] in/out; per draw (drghmc.py:348-389): partial momentum refresh, up to K attempts (retry test,
// proposal, accept test), unconditional momentum flip
extern "C" __global__ void __launch_bounds__(128) bk_user_drghmc(const bk::UserDrArgs a) {
    using namespace bk::user;
    const bk::UserRunArgs& ra = a.run;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ra.C) return;
    DrCtx ctx;
    ctx.params = reinterpret_cast<const T*>(ra.params);
    ctx.metric = reinterpret_cast<const T*>(ra.metric);
#pragma unroll
    for (int k = 0; k < bk::USER_DR_KMAX; ++k) {
        ctx.eps[k] = (T)a.eps[k];
        ctx.half[k] = (T)a.half_eps[k];
        ctx.cnt[k] = a.cnt[k];
    }
    ctx.prob_retry = a.prob_retry;
    const T s_keep = (T)a.s_keep, s_new = (T)a.s_new;
    T* row = reinterpret_cast<T*>(ra.theta) + c * (int64_t)D;
    T* rrow = reinterpret_cast<T*>(a.rho) + c * (int64_t)D;
    T th[D], rho[D], g[D];
    load_row(row, th);
    load_row(rrow, rho);
    T lp = log_density_gradient(th, g, ctx.params);
    for (int64_t t = 0; t < ra.n_draws; ++t) {
        T z[D];
        normals(ra, ra.C, c, t, z);
        T kin = T(0);
#pragma unroll
        for (int e = 0; e < D; ++e) {   // k_drg_refresh
            rho[e] = A::add(A::mul(rho[e], s_keep), A::mul(s_new, z[e]));
            kin = A::add(kin, A::mul(rho[e], dr_mg(ctx, e, rho[e])));
        }
        T cur_logp = A::sub(lp, A::mul(T(0.5), kin));
        T cur_hastings = T(0), reject_logp = T(0);
        int ui = 0;
        bool moved = false;
        for (int k = 0; k < a.K; ++k) {
            if (!(bk::log_u(uniform(ra, ra.C, c, t, ui++)) < dr_retry(ctx, reject_logp))) break;   // drghmc.py:369-371
            T qp[D], rp[D], gp[D], lpp;
            const T jp = trajectory(ctx, k, th, rho, g, qp, rp, gp, lpp);
            const T acc_lp = dr_accept<0>(k, ctx, qp, rp, gp, jp, cur_hastings, cur_logp);
            if (bk::log_u(uniform(ra, ra.C, c, t, ui++)) < acc_lp) {   // drghmc.py:378-381
#pragma unroll
                for (int e = 0; e < D; ++e) {
                    th[e] = qp[e];
                    rho[e] = rp[e];
                    g[e] = gp[e];
                }
                lp = lpp;
                cur_logp = jp;
                moved = true;
                break;
            }
            reject_logp = dr_log1m_exp(acc_lp);
            cur_hastings = A::add(cur_hastings, reject_logp);
        }
#pragma unroll
        for (int e = 0; e < D; ++e) rho[e] = -rho[e];   // drghmc.py:388
        emit(ra, c, t, th, cur_logp, moved);
        if (a.n_used) a.n_used[t * ra.C + c] = ui;
    }
#pragma unroll
    for (int e = 0; e < D; ++e) {
        row[e] = th[e];
        rrow[e] = rho[e];
    }
}

// ---- BK_PROGRAM_STRETCH: the Stretcher on a model, compiled on first use --------------------------------------------
#elif BK_PROGRAM == BK_PROGRAM_STRETCH

namespace bk {
namespace user {

// The generic engine stores (D - 1) log z, log p(q) and log p(theta) to memory before k_stretch_accept sums them.  Kept
// in registers, an fp32 sum with a product (the user's function may end in one) could be contracted into an FMA:
// these round every operation, as those stores do.  In fp64 they are Ar<double>'s.
__device__ __forceinline__ float rn_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float rn_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float rn_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double rn_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double rn_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double rn_sub(double a, double b) { return __dsub_rn(a, b); }

}  // namespace user
}  // namespace bk

// One half-step, one thread per active walker k: k_stretch_propose, the model's density of the proposal and
// k_stretch_accept (ensemble.cu) on the same uniforms and the same sequence of Ar<T> operations, with the proposal in
// registers.  Only the log density is used: the gradient the user's function writes is dead code after inlining.
extern "C" __global__ void __launch_bounds__(128) bk_user_stretch(const bk::UserStretchArgs a) {
    using namespace bk::user;
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.n) return;
    const T* params = reinterpret_cast<const T*>(a.params);
    T* row = reinterpret_cast<T*>(a.active) + k * (int64_t)D;
    T* lpk = reinterpret_cast<T*>(a.lp) + k;
    T th[D], q[D], unused[D];
    load_row(row, th);
    const T lp = a.eval_lp ? log_density_gradient(th, unused, params) : *lpk;
    int64_t j = (int64_t)(uniform(a, a.n, k, 0, 0) * (T)a.m);
    j = j < a.m ? j : a.m - 1;
    const T uz = A::add((T)a.lo, A::mul((T)a.width, uniform(a, a.n, k, 0, 1)));
    const T z = A::mul(uz, uz);
    const T* oj = reinterpret_cast<const T*>(a.other) + j * (int64_t)D;
#pragma unroll
    for (int e = 0; e < D; ++e) q[e] = A::add(oj[e], A::mul(z, A::sub(th[e], oj[e])));
    const T lpq = log_density_gradient(q, unused, params);
    const T log_q = rn_sub(rn_add(rn_mul((T)(D - 1), A::log_(z)), lpq), lp);
    const bool acc = bk::log_u(uniform(a, a.n, k, 0, 2)) < log_q;
    if (acc) {
#pragma unroll
        for (int e = 0; e < D; ++e) row[e] = q[e];
    }
    if (acc || a.eval_lp) *lpk = acc ? lpq : lp;
    if (a.accept) a.accept[k] = acc ? 1 : 0;
}

#endif  // BK_PROGRAM
#endif  // __CUDACC_RTC__
