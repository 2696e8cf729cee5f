// extern "C" entry points of the MCMC samplers: argument validation and the
// choice between the fused separable kernels and the generic engine.
#include <math.h>
#include <stdlib.h>

#include "dense_tc.h"
#include "sampler_generic.h"
#include "user_kernels.cuh"

using namespace bk;

bool bk::force_generic() {
    const char* e = getenv("BK_FORCE_GENERIC");
    return e && e[0] == '1';
}

namespace {

bool ptr_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int check_rng(const bk_rng* rng, const char* who) {
    BK_CHECK_ARG(rng, "%s: rng is required", who);
    BK_CHECK_ARG(rng->mode == BK_RNG_PHILOX || rng->mode == BK_RNG_INJECTED, "%s: bad rng mode %d",
                 who, rng->mode);
    if (rng->mode == BK_RNG_INJECTED)
        BK_CHECK_ARG(rng->normals && rng->uniforms && rng->n_uniform >= 1,
                     "%s: injected rng needs normals, uniforms and n_uniform >= 1", who);
    return BK_OK;
}

struct Common {
    const Model* m;
    int64_t C;
    int64_t n;
    const bk_rng* rng;
    bk_draw_out out;
};

template <typename T>
bool use_fused(const Model& m) { return m.separable() && m.d.dims <= SEP_MAX_D && !force_generic(); }

// user-written CUDA model with D <= USER_FUSED_MAX_D: one register-resident kernel per call (user_model.cu)
bool use_user_fused(const Model& m) { return user_fused(m) && !force_generic(); }

template <typename T>
void fill_sep(SepArgs<T>& a, const Model& m, void* theta, int64_t C, const void* metric, int64_t n,
              const bk_rng* rng, const bk_draw_out& out) {
    memset(&a, 0, sizeof(a));
    a.theta = (T*)theta;
    a.C = C;
    a.D = (int)m.d.dims;
    a.model.mu = (const T*)m.d.mu;
    a.model.prec = (const T*)m.d.prec;
    a.model.prec_scalar = (T)(1.0 / (m.d.sigma * m.d.sigma));
    a.model.metric = (const T*)metric;
    a.n_draws = n;
    a.rng = *rng;
    a.draws = (T*)out.draws;
    a.logp = (T*)out.logp;
    a.accept = out.accept;
    a.layout = out.layout;
    a.mom_mean = out.mom_mean;
    a.mom_m2 = out.mom_m2;
    a.mom_n0 = out.mom_n0;
    bool al = ptr_aligned16(theta) && ptr_aligned16(out.draws) && ptr_aligned16(m.d.mu) &&
              ptr_aligned16(m.d.prec) && ptr_aligned16(metric) &&
              (rng->mode != BK_RNG_INJECTED || ptr_aligned16(rng->normals));
    a.vec = (a.D % 4 == 0 && al) ? 1 : 0;
}

template <typename T>
void fill_gen(GenArgs<T>& p, const Model& m, void* theta, void* lp, void* grad, int64_t C,
              const void* metric, int64_t n, const bk_rng* rng, const bk_draw_out& out) {
    memset(&p, 0, sizeof(p));
    p.theta = (T*)theta;
    p.lp = (T*)lp;
    p.grad = (T*)grad;
    p.C = C;
    p.D = (int)m.d.dims;
    p.metric = (const T*)metric;
    p.n_draws = n;
    p.rng = *rng;
    p.draws = (T*)out.draws;
    p.logp = (T*)out.logp;
    p.accept = out.accept;
}

template <typename T>
int hmc_t(const Model& m, void* theta, void* lp, void* grad, int32_t* valid, int64_t C, double eps,
          int L, const void* metric, int64_t n, const bk_rng* rng, const bk_draw_out& out, void* ws,
          size_t wsb, cudaStream_t st) {
    if (use_fused<T>(m)) {
        SepArgs<T> a;
        fill_sep(a, m, theta, C, metric, n, rng, out);
        a.algo = ALGO_HMC;
        a.eps = (T)eps;
        a.half_eps = (T)(0.5 * eps);
        a.L = L;
        return launch_sep_sampler<T>(a, st);
    }
    if (use_user_fused(m)) {
        UserRunArgs a = user_args(m, theta, C, n, rng, out);
        a.metric = metric;
        a.eps = eps;
        a.half_eps = 0.5 * eps;
        a.L = L;
        return user_fused_sample(m, nullptr, ALGO_HMC, a, valid, st);
    }
    BK_CHECK_ARG(lp && grad, "bk_hmc_diag_sample: lp_cache/grad_cache are required for this model");
    if constexpr (sizeof(T) == 4) {
        // tensor-core pipeline: L-1 fused bf16 steps + one split-precision endpoint gradient
        if (dense_tc_enabled(m) && L >= 1)
            return dense_tc_hmc(m, (float*)theta, (float*)lp, (float*)grad, valid, C, eps, L,
                                (const float*)metric, n, rng, out, ws, wsb, st);
    }
    GenArgs<T> p;
    fill_gen(p, m, theta, lp, grad, C, metric, n, rng, out);
    p.eps = (T)eps;
    p.half_eps = (T)(0.5 * eps);
    p.L = L;
    return run_generic<T>(m, p, ALGO_HMC, valid, ws, wsb, st);
}

template <typename T>
int mala_t(const Model& m, void* theta, void* lp, void* grad, int32_t* valid, int64_t C, double eps,
           int64_t n, const bk_rng* rng, const bk_draw_out& out, void* ws, size_t wsb,
           cudaStream_t st) {
    const double sd = sqrt(2 * eps), coef = -0.25 / eps;  // mala.py:44, :79
    if (use_fused<T>(m)) {
        SepArgs<T> a;
        fill_sep(a, m, theta, C, nullptr, n, rng, out);
        a.algo = ALGO_MALA;
        a.eps = (T)eps;
        a.sd = (T)sd;
        a.coef = (T)coef;
        return launch_sep_sampler<T>(a, st);
    }
    if (use_user_fused(m)) {
        UserRunArgs a = user_args(m, theta, C, n, rng, out);
        a.eps = eps;
        a.sd = sd;
        a.coef = coef;
        return user_fused_sample(m, nullptr, ALGO_MALA, a, valid, st);
    }
    BK_CHECK_ARG(lp && grad, "bk_mala_sample: lp_cache/grad_cache are required for this model");
    if constexpr (sizeof(T) == 4) {
        // theta + eps g + sqrt(2 eps) z is one leapfrog step of size h = sqrt(2 eps) from momentum z,
        // and the Hastings ratio equals the Hamiltonian difference: begin -> split-precision
        // tcgen05 gradient -> accept, three launches per draw
        if (dense_tc_enabled(m))
            return dense_tc_hmc(m, (float*)theta, (float*)lp, (float*)grad, valid, C, sd, 1, nullptr, n, rng,
                                out, ws, wsb, st, /*report_lp=*/true);
    }
    GenArgs<T> p;
    fill_gen(p, m, theta, lp, grad, C, nullptr, n, rng, out);
    p.eps = (T)eps;
    p.sd = (T)sd;
    p.coef = (T)coef;
    return run_generic<T>(m, p, ALGO_MALA, valid, ws, wsb, st);
}

template <typename T>
int mh_t(const Model& m, void* theta, void* lp, int32_t* valid, int64_t C, double scale, int hastings,
         int64_t n, const bk_rng* rng, const bk_draw_out& out, void* ws, size_t wsb, cudaStream_t st) {
    if (use_fused<T>(m)) {
        SepArgs<T> a;
        fill_sep(a, m, theta, C, nullptr, n, rng, out);
        a.algo = ALGO_MHRW;
        a.scale = (T)scale;
        a.s2 = (T)(scale * scale);
        a.hastings = hastings;
        return launch_sep_sampler<T>(a, st);
    }
    if (use_user_fused(m)) {
        UserRunArgs a = user_args(m, theta, C, n, rng, out);
        a.scale = scale;
        a.s2 = scale * scale;
        a.hastings = hastings;
        return user_fused_sample(m, nullptr, ALGO_MHRW, a, valid, st);
    }
    BK_CHECK_ARG(lp, "bk_mh_rw_sample: lp_cache is required for this model");
    GenArgs<T> p;
    fill_gen(p, m, theta, lp, nullptr, C, nullptr, n, rng, out);
    p.scale = (T)scale;
    p.s2 = (T)(scale * scale);
    p.hastings = hastings;
    return run_generic<T>(m, p, ALGO_MHRW, valid, ws, wsb, st);
}

// ---- Metropolis / MetropolisHastings with a user proposal (bk_mh_cuda_*) ---------------------------------------------
// fused: one bk_user_mhp launch per call (user model, dims and n_normals <= USER_FUSED_MAX_D); otherwise the generic
// engine's ALGO_MHRW loop with bk_user_propose in place of k_mh_propose and its Hastings term in GenArgs::dh
bool use_mhp_fused(const Model& m, const UserProposal& p) { return user_mhp_fusable(m, p) && !force_generic(); }

// workspace of the three-launch path: [dh [C] | z, u scratch | generic engine]
size_t proposal_scratch_bytes(const Model& m, const UserProposal& p, int64_t C) {
    return align_up((size_t)C * (m.d.dtype == BK_F64 ? 8 : 4), 256) + user_propose_ws_bytes(p, C);
}

size_t mh_cuda_ws(const Model& m, const UserProposal& p, int64_t C) {
    if (C <= 0 || use_mhp_fused(m, p)) return 0;
    return proposal_scratch_bytes(m, p, C) +
           (m.d.dtype == BK_F64 ? generic_ws_bytes<double>(m, C) : generic_ws_bytes<float>(m, C));
}

struct ProposeCtx {
    const UserProposal* p;
    UserProposeArgs a;   // everything but theta, q, dh and t
};

int propose_hook(const void* ctx, const void* theta, void* q, void* dh, int64_t t, cudaStream_t st) {
    const ProposeCtx* h = static_cast<const ProposeCtx*>(ctx);
    UserProposeArgs a = h->a;
    a.theta = theta;
    a.q = q;
    a.dh = dh;
    a.t = t;
    return user_propose(*h->p, a, st);
}

template <typename T>
int mh_cuda_t(const Model& m, const UserProposal& pr, void* theta, void* lp, int32_t* valid, int64_t C, int hastings,
              int64_t n, const bk_rng* rng, const bk_draw_out& out, void* ws, size_t wsb, cudaStream_t st) {
    // Philox mode: the accept uniform is the single-uniform samplers' rule (philox_accept_uniform), which Row<T> and
    // user::accept_uniform apply only when n_uniform == 1; the proposal's own uniforms are TAG_UNIFORM words 0, 1, ...
    bk_rng r = *rng;
    if (r.mode == BK_RNG_PHILOX) r.n_uniform = 1;
    if (use_mhp_fused(m, pr)) {
        UserRunArgs a = user_args(m, theta, C, n, &r, out);
        a.hastings = hastings;
        a.prop_params = pr.params;
        return user_fused_sample(m, &pr, ALGO_MHRW, a, valid, st);
    }
    BK_CHECK_ARG(lp, "bk_mh_cuda_sample: lp_cache is required for this model");
    Arena ar(ws, wsb);
    T* dh = ar.take<T>(C);
    void* zbuf = ar.take<T>((size_t)C * pr.n_normals);
    void* ubuf = ar.take<T>((size_t)C * pr.n_uniforms);
    ar.off = align_up(ar.off, 256);
    const size_t gbytes = generic_ws_bytes<T>(m, C);
    if (!ar.ok() || wsb - ar.off < gbytes) {
        set_error("bk_mh_cuda_sample: workspace too small: need %zu bytes, got %zu", mh_cuda_ws(m, pr, C), wsb);
        return BK_E_WORKSPACE;
    }
    ProposeCtx ctx;
    memset(&ctx.a, 0, sizeof(ctx.a));
    ctx.p = &pr;
    ctx.a.params = pr.params;
    ctx.a.normals = r.normals;
    ctx.a.uniforms = r.uniforms;
    ctx.a.zbuf = zbuf;
    ctx.a.ubuf = ubuf;
    ctx.a.C = C;
    ctx.a.seed = r.seed;
    ctx.a.draw_offset = r.draw_offset;
    ctx.a.chain_offset = r.chain_offset;
    ctx.a.rng_mode = r.mode;
    ctx.a.n_uniform = r.n_uniform;
    const MhProposeHook hook{propose_hook, &ctx};
    GenArgs<T> p;
    fill_gen(p, m, theta, lp, nullptr, C, nullptr, n, &r, out);
    p.hastings = hastings;
    p.dh = hastings ? dh : nullptr;
    return run_generic<T>(m, p, ALGO_MHRW, valid, ar.base + ar.off, wsb - ar.off, st, &hook);
}

size_t sampler_ws(uint64_t h, int64_t C) {
    const Model* m = get_model(h);
    if (!m || C <= 0) return 0;
    if (m->separable() && m->d.dims <= SEP_MAX_D && !force_generic()) return 0;
    if (use_user_fused(*m)) return 0;
    if (dense_tc_enabled(*m)) {
        size_t a = dense_tc_hmc_ws_bytes(*m, C), b = generic_ws_bytes<float>(*m, C);
        return a > b ? a : b;
    }
    return m->d.dtype == BK_F64 ? generic_ws_bytes<double>(*m, C) : generic_ws_bytes<float>(*m, C);
}

// Streaming moments / series-major draws (bk_draw_out) are fused into the fp32 register-resident kernels; every
// other engine folds the draws it wrote in a second pass and cannot write the series-major layout.
// fused_extras: true when this call's engine handles bk_draw_out's extras itself.
bool fused_extras(const Model& m) { return m.d.dtype == BK_F32 && use_fused<float>(m); }

// the extras of an engine that writes [n, C, D] draws and folds the moments from them (check_folded / fold_extras)
int check_folded(const bk_draw_out& o, const char* who) {
    BK_CHECK_ARG(o.layout == BK_DRAWS_NCD || !o.draws,
                 "%s: the series-major draw layout is written by the fused fp32 separable samplers only", who);
    BK_CHECK_ARG(!o.mom_mean || o.draws, "%s: streaming moments on this engine fold the stored draws -- pass draws", who);
    return BK_OK;
}

int fold_extras(const Model& m, const bk_draw_out& o, int64_t C, int64_t n, void* stream) {
    if (!o.mom_mean) return BK_OK;
    return bk_moments_accumulate(o.draws, m.d.dtype, n, C * m.d.dims, o.mom_n0, o.mom_mean, o.mom_m2, stream);
}

int check_extras(const Model& m, const bk_draw_out& o, const char* who) {
    return fused_extras(m) ? BK_OK : check_folded(o, who);
}

int finish_extras(const Model& m, const bk_draw_out& o, int64_t C, int64_t n, void* stream) {
    return fused_extras(m) ? BK_OK : fold_extras(m, o, C, n, stream);
}

}  // namespace

namespace {
// out[c, :] = standard normals of global chain (chain_offset + c), Philox draw index `draw`, element blocks of 4 --
// the same (block, chain, draw) coordinates the samplers use, so initial states do not depend on the sharding
template <typename T>
__global__ void k_init_normal(T* __restrict__ out, int64_t C, int D, uint64_t seed, uint64_t chain_offset, uint32_t draw) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int nb = (D + 3) / 4;
    if (i >= C * nb) return;
    const int64_t c = i / nb;
    const int b = (int)(i % nb);
    T z[4];
    philox_normal4<T>(seed, (uint32_t)b, (uint32_t)(chain_offset + (uint64_t)c), draw, z);
    for (int k = 0; k < 4; ++k)
        if (4 * b + k < D) out[c * (int64_t)D + 4 * b + k] = z[k];
}
}  // namespace

extern "C" {

int bk_init_normal(void* out, int64_t C, int64_t D, int32_t dtype, uint64_t seed, uint64_t chain_offset, uint32_t draw,
                   void* stream) {
    BK_CHECK_ARG(out && C >= 0 && D >= 1, "bk_init_normal: bad argument");
    if (C == 0) return BK_OK;
    const int64_t n = C * ((D + 3) / 4);
    if (dtype == BK_F64)
        k_init_normal<double><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((double*)out, C, (int)D, seed,
                                                                                           chain_offset, draw);
    else
        k_init_normal<float><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((float*)out, C, (int)D, seed,
                                                                                          chain_offset, draw);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

size_t bk_hmc_diag_workspace_bytes(uint64_t h, int64_t C) { return sampler_ws(h, C); }
size_t bk_mala_workspace_bytes(uint64_t h, int64_t C) { return sampler_ws(h, C); }
size_t bk_mh_rw_workspace_bytes(uint64_t h, int64_t C) { return sampler_ws(h, C); }

int bk_hmc_diag_sample(uint64_t handle, void* theta, void* lp_cache, void* grad_cache,
                       int32_t* cache_valid_host, int64_t C, double stepsize, int32_t steps,
                       const void* metric, int64_t n_draws, const bk_rng* rng,
                       const bk_draw_out* out, void* ws, size_t ws_bytes, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && C >= 0 && n_draws >= 0, "bk_hmc_diag_sample: bad theta/C/n_draws");
    BK_CHECK_ARG(steps >= 0, "bk_hmc_diag_sample: steps must be >= 0 (got %d)", steps);
    int rc = check_rng(rng, "bk_hmc_diag_sample");
    if (rc) return rc;
    bk_draw_out o = out ? *out : bk_draw_out{nullptr, nullptr, nullptr};
    if (C == 0 || n_draws == 0) return BK_OK;
    if ((rc = check_extras(*m, o, "bk_hmc_diag_sample"))) return rc;
    if (m->d.dtype == BK_F64)
        rc = hmc_t<double>(*m, theta, lp_cache, grad_cache, cache_valid_host, C, stepsize, steps,
                             metric, n_draws, rng, o, ws, ws_bytes, (cudaStream_t)stream);
    else
        rc = hmc_t<float>(*m, theta, lp_cache, grad_cache, cache_valid_host, C, stepsize, steps, metric,
                        n_draws, rng, o, ws, ws_bytes, (cudaStream_t)stream);
    return rc ? rc : finish_extras(*m, o, C, n_draws, stream);
}

int bk_mala_sample(uint64_t handle, void* theta, void* lp_cache, void* grad_cache,
                   int32_t* cache_valid_host, int64_t C, double epsilon, int64_t n_draws,
                   const bk_rng* rng, const bk_draw_out* out, void* ws, size_t ws_bytes,
                   void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && C >= 0 && n_draws >= 0, "bk_mala_sample: bad theta/C/n_draws");
    BK_CHECK_ARG(epsilon > 0, "bk_mala_sample: epsilon must be > 0");
    int rc = check_rng(rng, "bk_mala_sample");
    if (rc) return rc;
    bk_draw_out o = out ? *out : bk_draw_out{nullptr, nullptr, nullptr};
    if (C == 0 || n_draws == 0) return BK_OK;
    if ((rc = check_extras(*m, o, "bk_mala_sample"))) return rc;
    if (m->d.dtype == BK_F64)
        rc = mala_t<double>(*m, theta, lp_cache, grad_cache, cache_valid_host, C, epsilon, n_draws,
                              rng, o, ws, ws_bytes, (cudaStream_t)stream);
    else
        rc = mala_t<float>(*m, theta, lp_cache, grad_cache, cache_valid_host, C, epsilon, n_draws, rng,
                         o, ws, ws_bytes, (cudaStream_t)stream);
    return rc ? rc : finish_extras(*m, o, C, n_draws, stream);
}

int bk_mh_rw_sample(uint64_t handle, void* theta, void* lp_cache, int32_t* cache_valid_host,
                    int64_t C, double scale, int32_t hastings, int64_t n_draws, const bk_rng* rng,
                    const bk_draw_out* out, void* ws, size_t ws_bytes, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && C >= 0 && n_draws >= 0, "bk_mh_rw_sample: bad theta/C/n_draws");
    BK_CHECK_ARG(scale > 0, "bk_mh_rw_sample: scale must be > 0");
    int rc = check_rng(rng, "bk_mh_rw_sample");
    if (rc) return rc;
    bk_draw_out o = out ? *out : bk_draw_out{nullptr, nullptr, nullptr};
    if (C == 0 || n_draws == 0) return BK_OK;
    if ((rc = check_extras(*m, o, "bk_mh_rw_sample"))) return rc;
    if (m->d.dtype == BK_F64)
        rc = mh_t<double>(*m, theta, lp_cache, cache_valid_host, C, scale, hastings, n_draws, rng, o,
                            ws, ws_bytes, (cudaStream_t)stream);
    else
        rc = mh_t<float>(*m, theta, lp_cache, cache_valid_host, C, scale, hastings, n_draws, rng, o, ws,
                       ws_bytes, (cudaStream_t)stream);
    return rc ? rc : finish_extras(*m, o, C, n_draws, stream);
}

size_t bk_mh_cuda_workspace_bytes(uint64_t model, uint64_t proposal, int64_t C) {
    const Model* m = get_model(model);
    const UserProposal* p = get_proposal(proposal);
    return m && p ? mh_cuda_ws(*m, *p, C) : 0;
}

int bk_mh_cuda_prepare(uint64_t model, uint64_t proposal, char* log_out, size_t log_bytes) {
    if (log_out && log_bytes) log_out[0] = '\0';
    const Model* m = get_model(model);
    if (!m) return BK_E_HANDLE;
    const UserProposal* p = get_proposal(proposal);
    if (!p) return BK_E_HANDLE;
    BK_CHECK_ARG(m->d.dims == p->dims && m->d.dtype == p->dtype,
                 "bk_mh_cuda_prepare: the proposal (dims %lld, dtype %d) does not match the model (dims %lld, dtype %d)",
                 (long long)p->dims, p->dtype, (long long)m->d.dims, m->d.dtype);
    return use_mhp_fused(*m, *p) ? user_mhp_prepare(*m, *p, "bk_mh_cuda_prepare", log_out, log_bytes) : BK_OK;
}

int bk_mh_cuda_sample(uint64_t model, uint64_t proposal, void* theta, void* lp_cache, int32_t* cache_valid_host,
                      int64_t C, int32_t hastings, int64_t n_draws, const bk_rng* rng, const bk_draw_out* out, void* ws,
                      size_t ws_bytes, void* stream) {
    const char* who = "bk_mh_cuda_sample";
    const Model* m = get_model(model);
    if (!m) return BK_E_HANDLE;
    const UserProposal* p = get_proposal(proposal);
    if (!p) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && C >= 0 && n_draws >= 0, "%s: bad theta/C/n_draws", who);
    BK_CHECK_ARG(m->d.dims == p->dims && m->d.dtype == p->dtype,
                 "%s: the proposal (dims %lld, dtype %d) does not match the model (dims %lld, dtype %d)", who,
                 (long long)p->dims, p->dtype, (long long)m->d.dims, m->d.dtype);
    BK_CHECK_ARG(!hastings || p->has_transition,
                 "%s: hastings needs a proposal created with has_transition = 1 (transition_log_density)", who);
    int rc = check_rng(rng, who);
    if (rc) return rc;
    if (rng->mode == BK_RNG_INJECTED)
        BK_CHECK_ARG(rng->n_uniform == 1 + p->n_uniforms,
                     "%s: injected rng needs n_uniform = 1 + the proposal's n_uniforms = %d (got %d)", who,
                     1 + p->n_uniforms, rng->n_uniform);
    bk_draw_out o = out ? *out : bk_draw_out{nullptr, nullptr, nullptr};
    if (C == 0 || n_draws == 0) return BK_OK;
    if ((rc = check_folded(o, who))) return rc;   // no engine of a user proposal fuses the extras
    if (m->d.dtype == BK_F64)
        rc = mh_cuda_t<double>(*m, *p, theta, lp_cache, cache_valid_host, C, hastings, n_draws, rng, o, ws, ws_bytes,
                               (cudaStream_t)stream);
    else
        rc = mh_cuda_t<float>(*m, *p, theta, lp_cache, cache_valid_host, C, hastings, n_draws, rng, o, ws, ws_bytes,
                              (cudaStream_t)stream);
    return rc ? rc : fold_extras(*m, o, C, n_draws, stream);
}

}  // extern "C"
