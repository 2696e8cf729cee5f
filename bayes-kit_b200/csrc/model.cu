// Model plugins: registry + batched log-density / gradient evaluation on
// CUDA cores (exact fp64 parity path and fp32 fallback).  The tcgen05 path for
// the dense-precision Gaussian lives in dense_tc.cu.
//
// Replaces the per-step Python callbacks model.log_density /
// log_density_gradient / log_prior / log_likelihood (typing.py:15-42; call
// sites hmc.py:38,45,50; mala.py:31,46; metropolis.py:99,119; smc.py:29-33).
#include <mutex>
#include <unordered_map>

#include "dense_tc.h"
#include "model.h"

namespace bk {

static std::mutex g_mu;
static std::unordered_map<uint64_t, Model> g_models;
static uint64_t g_next = 1;

const Model* get_model(uint64_t h) {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_models.find(h);
    if (it == g_models.end()) {
        set_error("unknown model handle %llu", (unsigned long long)h);
        return nullptr;
    }
    return &it->second;
}

int register_model(const Model& m, uint64_t* handle_out) {
    std::lock_guard<std::mutex> lk(g_mu);
    uint64_t h = g_next++;
    g_models[h] = m;
    *handle_out = h;
    return BK_OK;
}

// ---- elementwise models: one warp per chain --------------------------------
// kind ISO / DIAG / GAUSS_PRIOR_LIK (as a density: lik + prior)
template <typename T>
__global__ void k_sep_eval(int kind, const T* __restrict__ theta, int64_t C, int D, T prec_scalar,
                           const T* __restrict__ mu, const T* __restrict__ prec,
                           const T* __restrict__ m0, const T* __restrict__ p0, T* __restrict__ lp,
                           T* __restrict__ grad) {
    using A = Ar<T>;
    int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (c >= C) return;
    const T* x = theta + c * (int64_t)D;
    T s = T(0), s2 = T(0);
    for (int e = lane; e < D; e += 32) {
        T v = x[e], g;
        if (kind == BK_MODEL_ISO_GAUSS) {
            s = A::add(s, A::mul(v, v));
            g = -A::mul(prec_scalar, v);
        } else if (kind == BK_MODEL_DIAG_GAUSS) {
            T d = mu ? A::sub(v, mu[e]) : v;
            T pd = A::mul(prec[e], d);
            s = A::add(s, A::mul(d, pd));
            g = -pd;
        } else {  // GAUSS_PRIOR_LIK: lik + prior
            T dl = A::sub(v, mu[e]), dp = A::sub(v, m0[e]);
            s = A::add(s, A::mul(A::mul(prec[e], dl), dl));
            s2 = A::add(s2, A::mul(A::mul(p0[e], dp), dp));
            g = A::sub(-A::mul(prec[e], dl), A::mul(p0[e], dp));
        }
        if (grad) grad[c * (int64_t)D + e] = g;
    }
    s = warp_sum(s);
    s2 = warp_sum(s2);
    if (lane == 0) {
        if (kind == BK_MODEL_ISO_GAUSS) lp[c] = A::mul(T(-0.5), A::mul(prec_scalar, s));
        else if (kind == BK_MODEL_DIAG_GAUSS) lp[c] = A::mul(T(-0.5), s);
        else lp[c] = A::add(A::mul(T(-0.5), s), A::mul(T(-0.5), s2));
    }
}

template <typename T>
__global__ void k_prior_lik(const T* __restrict__ theta, int64_t C, int D, const T* __restrict__ mu,
                            const T* __restrict__ pl, const T* __restrict__ m0,
                            const T* __restrict__ p0, T* __restrict__ lprior, T* __restrict__ llik) {
    using A = Ar<T>;
    int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (c >= C) return;
    const T* x = theta + c * (int64_t)D;
    T s = T(0), s2 = T(0);
    for (int e = lane; e < D; e += 32) {
        T dl = A::sub(x[e], mu[e]), dp = A::sub(x[e], m0[e]);
        s = A::add(s, A::mul(A::mul(pl[e], dl), dl));
        s2 = A::add(s2, A::mul(A::mul(p0[e], dp), dp));
    }
    s = warp_sum(s);
    s2 = warp_sum(s2);
    if (lane == 0) {
        if (llik) llik[c] = A::mul(T(-0.5), s);
        if (lprior) lprior[c] = A::mul(T(-0.5), s2);
    }
}

// ---- beta-binomial on the logit scale (test/models/binomial.py:11-74), D = 1: one thread per chain
// p = inv_logit(theta); ll = log C(N,x) + x log p + (N-x) log(1-p); prior (with the logit Jacobian) =
// alpha log p + beta log(1-p) - log B(alpha, beta).  The gradient is analytic (the reference's test
// model differentiates numerically).
template <typename T>
__global__ void k_binom_eval(const T* __restrict__ theta, int64_t C, T al, T be, T xs, T Nn, T lch, T lbe,
                             T* __restrict__ lp, T* __restrict__ grad, T* __restrict__ lprior, T* __restrict__ llik) {
    using A = Ar<T>;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const T th = theta[c];
    const T e = A::exp_(-fabs(th)), l = A::log1p_(e);
    const T lp1 = th >= T(0) ? -l : A::sub(th, l), l1m = th >= T(0) ? A::sub(-th, l) : -l;
    const T p = th >= T(0) ? T(1) / A::add(T(1), e) : e / A::add(T(1), e);
    const T ll = A::add(A::add(lch, A::mul(xs, lp1)), A::mul(A::sub(Nn, xs), l1m));
    const T pr = A::sub(A::add(A::mul(al, lp1), A::mul(be, l1m)), lbe);
    if (lp) lp[c] = A::add(ll, pr);                                  // binomial.py:34-42
    if (grad) grad[c] = A::add(A::sub(xs, A::mul(Nn, p)), A::sub(al, A::mul(A::add(al, be), p)));
    if (lprior) lprior[c] = pr;
    if (llik) llik[c] = ll;
}

// ---- dense precision Gaussian on CUDA cores ----------------------------------
// out[c, j] = -sum_k (theta[c,k] - mu[k]) P[k, j]   (P symmetric, row-major)
// 64x64 tile, 16-wide k slabs, 256 threads, 4x4 micro-tile.
template <typename T>
__global__ void __launch_bounds__(256) k_dense_grad(const T* __restrict__ theta,
                                                    const T* __restrict__ mu,
                                                    const T* __restrict__ P, int64_t C, int D,
                                                    T* __restrict__ grad) {
    constexpr int BM = 64, BN = 64, BK = 16;
    __shared__ T As[BK][BM + 4];
    __shared__ T Bs[BK][BN + 4];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t row0 = (int64_t)blockIdx.y * BM;
    const int col0 = blockIdx.x * BN;
    T acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = T(0);
    for (int k0 = 0; k0 < D; k0 += BK) {
        // A slab: 64 rows x 16 k  (thread loads 4 elements)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int idx = threadIdx.x + 256 * i;  // 0..1023
            int r = idx >> 4, k = idx & 15;
            int64_t gr = row0 + r;
            int gk = k0 + k;
            T v = T(0);
            if (gr < C && gk < D) {
                v = theta[gr * (int64_t)D + gk];
                if (mu) v -= mu[gk];
            }
            As[k][r] = v;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int idx = threadIdx.x + 256 * i;
            int k = idx >> 6, c = idx & 63;
            int gk = k0 + k, gc = col0 + c;
            Bs[k][c] = (gk < D && gc < D) ? P[(int64_t)gk * D + gc] : T(0);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            T a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[k][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int64_t gr = row0 + ty * 4 + i;
        if (gr >= C) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int gc = col0 + tx * 4 + j;
            if (gc < D) grad[gr * (int64_t)D + gc] = -acc[i][j];
        }
    }
}

// lp[c] = 0.5 * (theta[c]-mu) . grad[c]     (= -0.5 r^T P r)
template <typename T>
__global__ void k_dense_lp(const T* __restrict__ theta, const T* __restrict__ mu,
                           const T* __restrict__ grad, int64_t C, int D, T* __restrict__ lp) {
    int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (c >= C) return;
    T s = T(0);
    for (int e = lane; e < D; e += 32) {
        T r = theta[c * (int64_t)D + e];
        if (mu) r -= mu[e];
        s = fma(r, grad[c * (int64_t)D + e], s);
    }
    s = warp_sum(s);
    if (lane == 0) lp[c] = T(0.5) * s;
}

template <typename T>
static int eval_t(const Model& m, const T* theta, int64_t C, T* lp, T* grad, void* ws,
                  size_t ws_bytes, cudaStream_t st, bool precise) {
    const int D = (int)m.d.dims;
    if (C == 0) return BK_OK;
    const unsigned wblocks = (unsigned)((C * 32 + 255) / 256);
    switch (m.d.kind) {
        case BK_MODEL_ISO_GAUSS:
        case BK_MODEL_DIAG_GAUSS:
        case BK_MODEL_GAUSS_PRIOR_LIK: {
            T ps = (T)(1.0 / (m.d.sigma * m.d.sigma));
            k_sep_eval<T><<<wblocks, 256, 0, st>>>(m.d.kind, theta, C, D, ps, (const T*)m.d.mu,
                                                    (const T*)m.d.prec, (const T*)m.d.m0,
                                                    (const T*)m.d.p0, lp, grad);
            BK_LAUNCH_CHECK();
            return BK_OK;
        }
        case BK_MODEL_DENSE_PREC_GAUSS: {
            T* g = grad;
            if (!g) {  // density only: gradient goes to scratch
                Arena ar(ws, ws_bytes);
                g = ar.take<T>((size_t)C * D);
                if (!ar.ok()) {
                    set_error("model eval workspace too small (%zu < %zu)", ws_bytes, ar.off);
                    return BK_E_WORKSPACE;
                }
            }
            if constexpr (sizeof(T) == 4) {
                if (dense_tc_enabled(m)) {  // tensor cores, 3-pass bf16 split (~2^-16 relative)
                    Arena ar2(ws, ws_bytes);
                    if (!grad) ar2.take<T>((size_t)C * D);
                    char* tws = ar2.take<char>(0);
                    int rc = dense_tc_grad(m, (const float*)theta, C, (float*)g, tws,
                                           ws_bytes > ar2.off ? ws_bytes - ar2.off : 0, st);
                    if (rc) return rc;
                    k_dense_lp<T><<<wblocks, 256, 0, st>>>(theta, (const T*)m.d.mu, g, C, D, lp);
                    BK_LAUNCH_CHECK();
                    return BK_OK;
                }
            }
            dim3 grid((D + 63) / 64, (unsigned)((C + 63) / 64));
            prof_begin(BK_PROF_GRAD, st);
            k_dense_grad<T><<<grid, 256, 0, st>>>(theta, (const T*)m.d.mu, (const T*)m.d.P, C, D, g);
            prof_end(BK_PROF_GRAD, st);
            BK_LAUNCH_CHECK();
            k_dense_lp<T><<<wblocks, 256, 0, st>>>(theta, (const T*)m.d.mu, g, C, D, lp);
            BK_LAUNCH_CHECK();
            return BK_OK;
        }
        case BK_MODEL_HIER_LOGREG:
            return hlr_eval(m, theta, C, lp, grad, ws, ws_bytes, st, precise);
        case BK_MODEL_BINOMIAL_LOGIT: {
            const double* q = m.d.scalars;
            k_binom_eval<T><<<(unsigned)((C + 255) / 256), 256, 0, st>>>(theta, C, (T)q[0], (T)q[1], (T)q[2], (T)q[3], (T)q[4],
                                                                        (T)q[5], lp, grad, (T*)nullptr, (T*)nullptr);
            BK_LAUNCH_CHECK();
            return BK_OK;
        }
        case BK_MODEL_USER_CUDA:
            return user_eval(m, theta, C, lp, grad, ws, ws_bytes, st);
        default:
            set_error("model kind %d has no device evaluator", m.d.kind);
            return BK_E_UNSUPPORTED;
    }
}

bool model_has_fast_path(const Model& m) { return hlr_tc_enabled(m); }

size_t model_eval_ws_bytes(const Model& m, int64_t C) {
    if (m.d.kind == BK_MODEL_HIER_LOGREG) return hlr_eval_ws_bytes(m, C);
    if (m.d.kind == BK_MODEL_DENSE_PREC_GAUSS) {
        size_t n = align_up((size_t)C * m.d.dims * (m.d.dtype == BK_F64 ? 8 : 4), 256) + 256;
        if (dense_tc_enabled(m)) n += 2 * align_up(align_up((size_t)C, 256) * m.Dp * 2, 256) + 512;  // bf16 hi/lo
        return n;
    }
    if (m.d.kind == BK_MODEL_USER_CUDA)   // gradient scratch of a density-only evaluation
        return align_up((size_t)C * m.d.dims * (m.d.dtype == BK_F64 ? 8 : 4), 256) + 256;
    return 0;
}

int model_eval(const Model& m, const void* theta, int64_t C, void* lp, void* grad, void* ws,
               size_t ws_bytes, cudaStream_t st, bool precise) {
    if (m.d.dtype == BK_F64)
        return eval_t<double>(m, (const double*)theta, C, (double*)lp, (double*)grad, ws, ws_bytes, st, true);
    return eval_t<float>(m, (const float*)theta, C, (float*)lp, (float*)grad, ws, ws_bytes, st, precise);
}

}  // namespace bk

using namespace bk;

extern "C" {

size_t bk_model_workspace_bytes(const bk_model_desc* desc) {
    if (!desc) return 0;
    return 256 + dense_tc_model_ws_bytes(*desc) + hlr_tc_model_ws_bytes(*desc);  // tensor-core operands
}

int bk_model_create(const bk_model_desc* desc, void* ws, size_t ws_bytes, void* stream,
                    uint64_t* handle_out) {
    BK_CHECK_ARG(desc && handle_out, "bk_model_create: null argument");
    BK_CHECK_ARG(desc->dtype == BK_F32 || desc->dtype == BK_F64, "bk_model_create: bad dtype %d",
                 desc->dtype);
    BK_CHECK_ARG(desc->dims >= 1, "bk_model_create: dims must be >= 1 (got %lld)",
                 (long long)desc->dims);
    switch (desc->kind) {
        case BK_MODEL_ISO_GAUSS:
            BK_CHECK_ARG(desc->sigma > 0, "ISO_GAUSS: sigma must be > 0");
            break;
        case BK_MODEL_DIAG_GAUSS:
            BK_CHECK_ARG(desc->prec, "DIAG_GAUSS: prec is required");
            break;
        case BK_MODEL_DENSE_PREC_GAUSS:
            BK_CHECK_ARG(desc->P, "DENSE_PREC_GAUSS: P is required");
            break;
        case BK_MODEL_GAUSS_PRIOR_LIK:
            BK_CHECK_ARG(desc->mu && desc->prec && desc->m0 && desc->p0,
                         "GAUSS_PRIOR_LIK: mu, prec, m0, p0 are required");
            break;
        case BK_MODEL_HIER_LOGREG:
            BK_CHECK_ARG(desc->X && desc->y && desc->n_obs > 0, "HIER_LOGREG: X, y, n_obs required");
            BK_CHECK_ARG(desc->dims >= 3, "HIER_LOGREG: dims = Dx + 2 must be >= 3");
            break;
        case BK_MODEL_BINOMIAL_LOGIT:
            BK_CHECK_ARG(desc->dims == 1, "BINOMIAL_LOGIT: dims must be 1");
            BK_CHECK_ARG(desc->scalars[0] > 0 && desc->scalars[1] > 0, "BINOMIAL_LOGIT: alpha, beta must be > 0");
            BK_CHECK_ARG(desc->scalars[3] >= desc->scalars[2] && desc->scalars[2] >= 0, "BINOMIAL_LOGIT: need 0 <= x <= N");
            break;
        case BK_MODEL_USER_CUDA:
            set_error("bk_model_create: USER_CUDA models are created by bk_model_create_cuda");
            return BK_E_INVALID;
        default:
            set_error("bk_model_create: unknown kind %d", desc->kind);
            return BK_E_INVALID;
    }
    Model m;
    m.d = *desc;
    if (m.d.kind != BK_MODEL_ISO_GAUSS) m.d.sigma = 1.0;
    if (ws && ws_bytes >= dense_tc_model_ws_bytes(*desc) && dense_tc_model_ws_bytes(*desc) > 0) {
        int rc = dense_tc_prepare(m, ws, ws_bytes, (cudaStream_t)stream);
        if (rc) return rc;
    }
    if (ws && ws_bytes >= hlr_tc_model_ws_bytes(*desc) && hlr_tc_model_ws_bytes(*desc) > 0) {
        int rc = hlr_tc_prepare(m, ws, ws_bytes, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return register_model(m, handle_out);
}

int bk_model_destroy(uint64_t handle) {
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_models.erase(handle)) {
        set_error("bk_model_destroy: unknown handle");
        return BK_E_HANDLE;
    }
    return BK_OK;
}

int64_t bk_model_dims(uint64_t handle) {
    const Model* m = get_model(handle);
    return m ? m->d.dims : -1;
}

size_t bk_model_eval_workspace_bytes(uint64_t handle, int64_t C) {
    const Model* m = get_model(handle);
    return m ? model_eval_ws_bytes(*m, C) : 0;
}

int bk_model_log_density_gradient(uint64_t handle, const void* theta, int64_t C, void* lp_out,
                                  void* grad_out, void* ws, size_t ws_bytes, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && lp_out && C >= 0, "bk_model_log_density_gradient: bad argument");
    return model_eval(*m, theta, C, lp_out, grad_out, ws, ws_bytes, (cudaStream_t)stream);
}

int bk_model_log_density_gradient_fast(uint64_t handle, const void* theta, int64_t C, void* lp_out,
                                       void* grad_out, void* ws, size_t ws_bytes, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(theta && lp_out && C >= 0, "bk_model_log_density_gradient_fast: bad argument");
    return model_eval(*m, theta, C, lp_out, grad_out, ws, ws_bytes, (cudaStream_t)stream, /*precise=*/false);
}

int bk_model_log_prior_likelihood(uint64_t handle, const void* theta, int64_t C,
                                  void* log_prior_out, void* log_lik_out, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(m->d.kind == BK_MODEL_GAUSS_PRIOR_LIK || m->d.kind == BK_MODEL_BINOMIAL_LOGIT || user_prior_lik(*m),
                 "log_prior/log_likelihood need a GAUSS_PRIOR_LIK or BINOMIAL_LOGIT model, or a user model created by "
                 "bk_model_create_cuda_prior_lik");
    if (C == 0) return BK_OK;
    if (m->d.kind == BK_MODEL_USER_CUDA)
        return user_log_prior_likelihood(*m, theta, C, log_prior_out, log_lik_out, (cudaStream_t)stream);
    const int D = (int)m->d.dims;
    const unsigned blocks = (unsigned)((C * 32 + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (m->d.kind == BK_MODEL_BINOMIAL_LOGIT) {
        const double* q = m->d.scalars;
        const unsigned bb = (unsigned)((C + 255) / 256);
        if (m->d.dtype == BK_F64)
            k_binom_eval<double><<<bb, 256, 0, st>>>((const double*)theta, C, q[0], q[1], q[2], q[3], q[4], q[5], nullptr,
                                                      nullptr, (double*)log_prior_out, (double*)log_lik_out);
        else
            k_binom_eval<float><<<bb, 256, 0, st>>>((const float*)theta, C, (float)q[0], (float)q[1], (float)q[2], (float)q[3],
                                                     (float)q[4], (float)q[5], nullptr, nullptr, (float*)log_prior_out,
                                                     (float*)log_lik_out);
        BK_LAUNCH_CHECK();
        return BK_OK;
    }
    if (m->d.dtype == BK_F64)
        k_prior_lik<double><<<blocks, 256, 0, st>>>((const double*)theta, C, D, (const double*)m->d.mu,
                                                     (const double*)m->d.prec, (const double*)m->d.m0,
                                                     (const double*)m->d.p0, (double*)log_prior_out,
                                                     (double*)log_lik_out);
    else
        k_prior_lik<float><<<blocks, 256, 0, st>>>((const float*)theta, C, D, (const float*)m->d.mu,
                                                    (const float*)m->d.prec, (const float*)m->d.m0,
                                                    (const float*)m->d.p0, (float*)log_prior_out,
                                                    (float*)log_lik_out);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

}  // extern "C"
