#pragma once
#include "model.h"
#include "sampler_sep.h"

namespace bk {

template <typename T>
struct GenArgs {
    // state (caller buffers)
    T* theta;  // [C, D]
    T* lp;     // [C]   log p(theta)
    T* grad;   // [C, D] grad log p(theta)   (unused by MHRW)
    // workspace (carved by run_generic)
    T *q, *r, *grad_q, *lp_q, *h0;
    int64_t C;
    int D;
    const T* metric;
    T eps, half_eps;
    int L;
    T sd, coef;
    T scale, s2;
    int hastings;
    int64_t n_draws;
    bk_rng rng;
    T* draws;
    T* logp;
    int32_t* accept;
    T* dh;      // [C] Hastings term of a user proposal (log q(theta | q) - log q(q | theta)), added by k_mh_accept in
                // place of the Gaussian random walk's; NULL: the built-in term (when hastings)
};

// Replaces k_mh_propose in run_generic's ALGO_MHRW loop (user proposals): writes q [C, D] from theta [C, D] (and, for
// a gradient proposal, grad [C, D] = grad log p(theta)) for draw t of the call, and dh [C] when dh is not NULL.
// A gradient proposal (hastings not NULL) writes its forward term to dh; after the model's evaluation of q with its
// gradient grad_q, hastings replaces it by the Hastings term.  The loop then keeps grad valid with lp.
struct MhProposeHook {
    int (*fn)(const void* ctx, const void* theta, const void* grad, void* q, void* dh, int64_t t, cudaStream_t st);
    const void* ctx;
    bool gradient = false;
    int (*hastings)(const void* ctx, const void* theta, const void* q, const void* grad_q, void* dh,
                    cudaStream_t st) = nullptr;
};

template <typename T>
size_t generic_ws_bytes(const Model& m, int64_t C);
template <typename T>
int run_generic(const Model& m, GenArgs<T> p, int algo, int* cache_valid, void* ws, size_t ws_bytes,
                cudaStream_t st, const MhProposeHook* propose = nullptr);

}  // namespace bk
