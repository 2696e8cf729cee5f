// Affine-invariant ensemble "stretch move" (Goodman & Weare 2010), the algorithm sketched in the
// reference's ensemble.py:16-66 (commented out upstream: parity is pinned by oracle/samplers.py only).
//
// One call updates the n ACTIVE walkers against the m walkers of the COMPLEMENTARY half:
//   j ~ U{0..m-1};  z = u_z^2, u_z ~ U(1/sqrt a, sqrt a)          (ensemble.py:43-46, 55)
//   theta* = other[j] + z (theta_k - other[j])                      (:50)
//   accept iff log u < (D-1) log z + log p(theta*) - log p(theta_k) (:51-53)
// Every active walker moves in parallel -- that is the point of splitting the ensemble.  Three
// launches: propose (warp per walker), the plugin's batched density (tensor cores where it has
// them), accept.  A user model (bk_model_create_cuda*) with dims <= USER_FUSED_MAX_D runs all three
// in one launch of the runtime-compiled bk_user_stretch (user_model.cu, one thread per walker).  The
// current walkers' log densities are cached (the reference's TODO, :69); both engines keep the cache.
#include "model.h"
#include "sep_common.cuh"

namespace bk {

template <typename T>
struct StretchArgs {
    T* active;           // [n, D] in/out
    T* lp;               // [n] cached log p(active), in/out
    const T* other;      // [m, D]
    T* prop;             // [n, D] workspace
    T* lp_prop;          // [n]
    T* logz;             // [n]  (D - 1) log z
    int64_t n, m;
    int D;
    T lo, width;         // u_z = lo + width * u,  lo = 1/sqrt(a), width = sqrt(a) - 1/sqrt(a)
    bk_rng rng;          // Philox: chain_offset = global id of active[0]; injected: uniforms [n, 3]
    int32_t* accept;
};

template <typename T>
__device__ __forceinline__ T stretch_uniform(const bk_rng& rng, int64_t k, int which) {
    if (rng.mode == BK_RNG_INJECTED) return reinterpret_cast<const T*>(rng.uniforms)[k * 3 + which];
    return philox_uniform<T>(rng.seed, (uint32_t)which, (uint32_t)(rng.chain_offset + (uint64_t)k),
                             (uint32_t)rng.draw_offset);
}

template <typename T>
__global__ void k_stretch_propose(StretchArgs<T> a) {
    using A = Ar<T>;
    const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= a.n) return;
    int64_t j = (int64_t)(stretch_uniform<T>(a.rng, k, 0) * (T)a.m);
    j = j < a.m ? j : a.m - 1;
    const T uz = A::add(a.lo, A::mul(a.width, stretch_uniform<T>(a.rng, k, 1)));
    const T z = A::mul(uz, uz);
    const T* tk = a.active + k * (int64_t)a.D;
    const T* tj = a.other + j * (int64_t)a.D;
    T* pr = a.prop + k * (int64_t)a.D;
    for (int e = lane; e < a.D; e += 32) pr[e] = A::add(tj[e], A::mul(z, A::sub(tk[e], tj[e])));
    if (lane == 0) a.logz[k] = A::mul((T)(a.D - 1), A::log_(z));
}

template <typename T>
__global__ void k_stretch_accept(StretchArgs<T> a) {
    using A = Ar<T>;
    const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (k >= a.n) return;
    const T log_q = A::sub(A::add(a.logz[k], a.lp_prop[k]), a.lp[k]);
    const bool acc = log_u(stretch_uniform<T>(a.rng, k, 2)) < log_q;
    if (acc) {
        T* tk = a.active + k * (int64_t)a.D;
        const T* pr = a.prop + k * (int64_t)a.D;
        for (int e = lane; e < a.D; e += 32) tk[e] = pr[e];
    }
    if (lane == 0) {
        if (acc) a.lp[k] = a.lp_prop[k];
        if (a.accept) a.accept[k] = acc ? 1 : 0;
    }
}

template <typename T>
static int stretch_t(const Model& m, void* active, void* lp, int32_t* lp_valid, const void* other, int64_t n,
                     int64_t mo, double a, const bk_rng* rng, int32_t* accept, void* ws, size_t ws_bytes,
                     cudaStream_t st) {
    const int D = (int)m.d.dims;
    Arena ar(ws, ws_bytes);
    StretchArgs<T> s;
    memset(&s, 0, sizeof(s));
    s.prop = ar.take<T>((size_t)n * D);
    s.lp_prop = ar.take<T>((size_t)n);
    s.logz = ar.take<T>((size_t)n);
    const size_t ebytes = model_eval_ws_bytes(m, n);
    void* ews = ar.take<char>(ebytes);
    if (!ar.ok()) {
        set_error("bk_stretch_move: workspace too small (need %zu bytes, got %zu)", ar.off, ws_bytes);
        return BK_E_WORKSPACE;
    }
    int rc;
    if (!lp_valid || !*lp_valid) {
        if ((rc = model_eval(m, active, n, lp, nullptr, ews, ebytes, st))) return rc;
        if (lp_valid) *lp_valid = 1;
    }
    s.active = (T*)active; s.lp = (T*)lp; s.other = (const T*)other; s.n = n; s.m = mo; s.D = D;
    s.lo = (T)(1.0 / sqrt(a)); s.width = (T)(sqrt(a) - 1.0 / sqrt(a));
    s.rng = *rng; s.accept = accept;
    const unsigned blocks = (unsigned)((n * 32 + 255) / 256);
    k_stretch_propose<T><<<blocks, 256, 0, st>>>(s);
    BK_LAUNCH_CHECK();
    if ((rc = model_eval(m, s.prop, n, s.lp_prop, nullptr, ews, ebytes, st))) return rc;
    k_stretch_accept<T><<<blocks, 256, 0, st>>>(s);
    BK_LAUNCH_CHECK();
    return BK_OK;
}

}  // namespace bk

using namespace bk;

// the runtime-compiled bk_user_stretch serves user models up to USER_FUSED_MAX_D dims; every other model runs stretch_t
static bool stretch_user_fused(const Model& m) { return !force_generic() && user_fused(m); }

extern "C" {

size_t bk_stretch_workspace_bytes(uint64_t handle, int64_t n_active) {
    const Model* m = get_model(handle);
    if (!m || n_active <= 0) return 256;
    if (stretch_user_fused(*m)) return 0;
    const size_t es = m->d.dtype == BK_F64 ? 8 : 4;
    return align_up((size_t)n_active * m->d.dims * es, 256) + 2 * align_up((size_t)n_active * es, 256) +
           model_eval_ws_bytes(*m, n_active) + 1024;
}

int bk_stretch_cuda_prepare(uint64_t handle, char* log_out, size_t log_bytes) {
    if (log_out && log_bytes) log_out[0] = '\0';
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    return stretch_user_fused(*m) ? user_stretch_prepare(*m, log_out, log_bytes) : BK_OK;
}

int bk_stretch_move(uint64_t handle, void* active, void* lp_active, int32_t* lp_valid_host, const void* other,
                    int64_t n_active, int64_t n_other, double a, const bk_rng* rng, int32_t* accept_out,
                    void* ws, size_t ws_bytes, void* stream) {
    const Model* m = get_model(handle);
    if (!m) return BK_E_HANDLE;
    BK_CHECK_ARG(active && lp_active && other && rng, "bk_stretch_move: null argument");
    BK_CHECK_ARG(n_active >= 0 && n_other >= 1, "bk_stretch_move: need n_active >= 0 and n_other >= 1");
    BK_CHECK_ARG(a >= 1.0, "stretch bound must be greater than or equal to 1; found a=%g", a);
    BK_CHECK_ARG(rng->mode == BK_RNG_PHILOX || (rng->mode == BK_RNG_INJECTED && rng->uniforms),
                 "bk_stretch_move: injected rng needs uniforms [n_active, 3]");
    if (n_active == 0) return BK_OK;
    if (stretch_user_fused(*m)) {
        const bool eval_lp = !lp_valid_host || !*lp_valid_host;
        if (int rc = user_stretch_move(*m, active, lp_active, eval_lp, other, n_active, n_other, a, rng, accept_out,
                                       (cudaStream_t)stream))
            return rc;
        if (lp_valid_host) *lp_valid_host = 1;
        return BK_OK;
    }
    if (m->d.dtype == BK_F64)
        return stretch_t<double>(*m, active, lp_active, lp_valid_host, other, n_active, n_other, a, rng, accept_out,
                                 ws, ws_bytes, (cudaStream_t)stream);
    return stretch_t<float>(*m, active, lp_active, lp_valid_host, other, n_active, n_other, a, rng, accept_out, ws,
                            ws_bytes, (cudaStream_t)stream);
}

}  // extern "C"
