/*
 * bk.h -- C ABI of libbk_b200.so: the B200-native (sm_100a) replacement for the
 * data-parallel sampling hot path of flatironinstitute/bayes-kit.
 *
 * The reference has NO FFI layer: its boundary is a pair of Python structural
 * protocols (bayes_kit/typing.py:15-42) called once per gradient from the
 * interpreter.  This header is what a reference-side binding (ctypes, see
 * INTEGRATION.md) binds instead.  Every entry point names the reference
 * function(s) it replaces.
 *
 * Conventions
 *   - extern "C", plain C types only; no torch / CUDA types in signatures
 *     (`stream` is a cudaStream_t passed as void*; 0 = default stream).
 *   - every function returns int: 0 = BK_OK, <0 = BK_E_*; bk_last_error()
 *     gives the thread-local message.
 *   - the CALLER owns every buffer.  All pointers are DEVICE pointers unless
 *     a name ends in _host.  The library never frees caller memory and
 *     allocates no device memory: scratch is passed in (`ws`, sized by the
 *     matching *_workspace_bytes()).  One exception: bk_model_create_cuda loads
 *     the module it compiles (kept for the life of the process).
 *   - all work is enqueued asynchronously on `stream`; no hidden syncs.
 *   - tensors are dense row-major: theta [C, D], draws [n, C, D].
 *   - `dtype`: BK_F32 (timed mode) or BK_F64 (parity mode: separate
 *     multiply/add roundings in NumPy's association order).
 */
#ifndef BK_B200_H
#define BK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BK_ABI_VERSION 1

#if defined(__GNUC__)
#define BK_API __attribute__((visibility("default")))
#else
#define BK_API
#endif

enum { BK_OK = 0, BK_E_INVALID = -1, BK_E_UNSUPPORTED = -2, BK_E_CUDA = -3,
       BK_E_WORKSPACE = -4, BK_E_HANDLE = -5 };

enum { BK_F32 = 0, BK_F64 = 1 };

/* model plugin kinds (device-side log density + gradient; replaces the Python
 * callbacks model.log_density / log_density_gradient / log_prior /
 * log_likelihood, typing.py:15-42) */
enum { BK_MODEL_ISO_GAUSS = 0,        /* -0.5 |theta|^2 / sigma^2                          */
       BK_MODEL_DIAG_GAUSS = 1,       /* -0.5 sum prec_i (theta_i - mu_i)^2                */
       BK_MODEL_DENSE_PREC_GAUSS = 2, /* -0.5 (theta-mu)^T P (theta-mu)                    */
       BK_MODEL_HIER_LOGREG = 3,      /* hierarchical logistic regression (DESIGN.md)      */
       BK_MODEL_GAUSS_PRIOR_LIK = 4,  /* prior N(m0, 1/p0) x likelihood N(mu, 1/pl) (SMC)  */
       BK_MODEL_BINOMIAL_LOGIT = 5,   /* beta-binomial on the logit scale, D = 1: the reference's own
                                         test target (test/models/binomial.py:11-74), with
                                         log_prior / log_likelihood for the SMC                */
       BK_MODEL_USER_CUDA = 6         /* user-written CUDA source, bk_model_create_cuda        */ };

enum { BK_RNG_PHILOX = 0,   /* device Philox4x32-10, counter = (block, tag, chain, draw) */
       BK_RNG_INJECTED = 1  /* pre-drawn streams in the reference's consumption order */ };

enum { BK_RESAMPLE_MULTINOMIAL = 0, /* smc.py:64-75 (legacy np.random.choice)           */
       BK_RESAMPLE_SYSTEMATIC = 1   /* north_star item 2; log-sum-exp normalised        */ };

enum { BK_IAT_IPSE = 0, BK_IAT_IMSE = 1 };

typedef struct bk_model_desc {
    int32_t kind;        /* BK_MODEL_*                                                  */
    int32_t dtype;       /* dtype of every array below                                  */
    int64_t dims;        /* D (HIER_LOGREG: Dx + 2)                                     */
    double  sigma;       /* ISO_GAUSS                                                   */
    const void* mu;      /* [D] DIAG/DENSE mean (NULL = 0); GAUSS_PRIOR_LIK lik. mean    */
    const void* prec;    /* [D] DIAG precisions;            GAUSS_PRIOR_LIK lik. prec    */
    const void* P;       /* [D, D] DENSE precision, row-major, symmetric                 */
    const void* m0;      /* [D] GAUSS_PRIOR_LIK prior mean                               */
    const void* p0;      /* [D] GAUSS_PRIOR_LIK prior precisions                         */
    const void* X;       /* [N, Dx] HIER_LOGREG design matrix                            */
    const void* y;       /* [N] HIER_LOGREG 0/1 responses                                */
    int64_t n_obs;       /* N                                                            */
    double  scalars[8];  /* BINOMIAL_LOGIT: alpha, beta, x, N, log C(N, x), log B(alpha, beta)      */
} bk_model_desc;

typedef struct bk_rng {
    int32_t  mode;          /* BK_RNG_*                                                  */
    int32_t  n_uniform;     /* INJECTED: uniforms per (draw, chain) (1; 2K for DrGHMC)   */
    uint64_t seed;          /* PHILOX key                                                */
    uint64_t draw_offset;   /* PHILOX: index of this call's first draw                   */
    uint64_t chain_offset;  /* PHILOX: global id of local chain 0 (multi-GPU shards)     */
    const void* normals;    /* INJECTED: [n_draws, C, D] standard normals (dtype)        */
    const void* uniforms;   /* INJECTED: [n_draws, C, n_uniform] uniforms in [0,1)       */
} bk_rng;
/* bk_mh_cuda_sample (user proposals) reads INJECTED streams as normals [n_draws, C, n_normals] and uniforms
 * [n_draws, C, 1 + n_uniforms] (n_uniform = 1 + n_uniforms): column 0 is the accept uniform, column 1 + k the
 * proposal's u[k].  In PHILOX mode z[k] is element k % 4 of the normals of element block b(k) = k / 4, or k / 4 + 1
 * from block ceil(D / 4) on (that block holds the accept uniform of the single-uniform samplers, which is unchanged;
 * with n_normals <= D, z is exactly the random walk's normal vector), and u[k] is the k-th TAG_UNIFORM uniform.
 * The SMC's proposal move (BK_SMC_KERNEL_PROPOSAL) uses the same layout with the particle in place of the chain and
 * the temperature step n in place of the draw: INJECTED normals [M_local, n_normals] and uniforms
 * [M_local, 1 + n_uniforms]; PHILOX z and u of (chain_offset + m, n) by the rule above, the accept uniform of
 * (chain_offset + m, n) by the random-walk move's rule. */

enum { BK_DRAWS_NCD = 0,  /* draws [n_draws, C, D]: one draw of every chain after the other      */
       BK_DRAWS_CDN = 1   /* draws [C, D, n_draws]: every (chain, dim) SERIES contiguous over the
                             draws -- what bk_iat_ess / bk_autocorr stream without a transposition
                             (SURVEY 8(f)-2); fused separable samplers only                      */ };

/* per-call outputs shared by the MCMC samplers; any pointer may be NULL */
typedef struct bk_draw_out {
    void*    draws;   /* [n_draws, C, D] (or [C, D, n_draws], see layout)                */
    void*    logp;    /* [n_draws, C] value sample() returns (HMC/DrGHMC: JOINT logp)    */
    int32_t* accept;  /* [n_draws, C] 1 = proposal accepted                              */
    int32_t  layout;  /* BK_DRAWS_*                                                      */
    /* Streaming moments folded in the sampler's epilogue (SURVEY 8(f)-2): running per-chain,
     * per-dimension mean [C, D] and sum of squared deviations M2 [C, D] (fp64) that already cover
     * mom_n0 draws are updated with this call's n_draws WITHOUT a pass over stored draws (the fused
     * separable samplers accumulate in registers across the draws of the launch and merge once, Chan et
     * al.); the other engines fold the draws they wrote (draws must be given).  NULL: off. */
    double*  mom_mean;
    double*  mom_m2;
    int64_t  mom_n0;
} bk_draw_out;

BK_API const char* bk_last_error(void);
BK_API int bk_abi_version(void);
/* number of kernels launched by this process through the library so far */
BK_API uint64_t bk_launch_count(void);

/* Optional in-library CUDA-event timing of the dominant kernels, recorded on
 * the launch stream (bench.py's live roofline measurement).  bk_profile_read
 * synchronises the recorded events, returns the summed device time and launch
 * count of `tag` since the last read, and resets that tag. */
enum { BK_PROF_GRAD = 0,      /* model gradient kernel (dense plugin: GEMM, tcgen05 GRAD mode) */
       BK_PROF_SAMPLER = 1,   /* fused sampler kernel                                          */
       BK_PROF_STEP = 2,      /* tcgen05 GEMM with the fused leapfrog epilogue (STEP mode)     */
       BK_PROF_NTAGS = 4 };
BK_API int bk_profile_enable(int32_t on);
BK_API int bk_profile_read(int32_t tag, double* total_ms_out, uint64_t* launches_out);

/* ---- model plugins (typing.py:15-42) ------------------------------------ */
BK_API size_t bk_model_workspace_bytes(const bk_model_desc* desc);
/* `ws` (device, bk_model_workspace_bytes) holds derived operands (bf16 splits
 * of P, P*mu, ...) and must outlive the handle. */
BK_API int bk_model_create(const bk_model_desc* desc, void* ws, size_t ws_bytes, void* stream,
                    uint64_t* handle_out);
BK_API int bk_model_destroy(uint64_t handle);
BK_API int64_t bk_model_dims(uint64_t handle);
BK_API size_t bk_model_eval_workspace_bytes(uint64_t handle, int64_t C);
/* model.log_density / log_density_gradient, batched: theta [C,D] -> lp [C],
 * grad [C,D] (grad may be NULL).  hmc.py:38,45,50; mala.py:31,46 */
BK_API int bk_model_log_density_gradient(uint64_t handle, const void* theta, int64_t C, void* lp_out,
                                  void* grad_out, void* ws, size_t ws_bytes, void* stream);
/* Same contract, but the plugin may answer with its reduced-precision tensor-core path
 * (bf16 operands, fp32 accumulate).  This is what the samplers use for INTERIOR leapfrog
 * gradients -- any deterministic gradient keeps the leapfrog map reversible and volume
 * preserving; everything that enters a Metropolis test uses the precise evaluation above. */
BK_API int bk_model_log_density_gradient_fast(uint64_t handle, const void* theta, int64_t C,
                                       void* lp_out, void* grad_out, void* ws, size_t ws_bytes,
                                       void* stream);
/* log_prior / log_likelihood (smc.py:29-33): GAUSS_PRIOR_LIK, BINOMIAL_LOGIT, and user models created by
 * bk_model_create_cuda_prior_lik.  Either output may be NULL. */
BK_API int bk_model_log_prior_likelihood(uint64_t handle, const void* theta, int64_t C,
                                  void* log_prior_out, void* log_lik_out, void* stream);

/* User-written model (BK_MODEL_USER_CUDA): any log density the caller can write as one CUDA C++ function
 *
 *     __device__ bk_real log_density_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
 *
 * returning log p(theta) and writing d log p / d theta into grad[0 .. BK_DIMS).  bk_real is float (BK_F32) or
 * double (BK_F64), BK_DIMS the model's dimension as a compile-time constant; helper functions, structs and
 * constants may precede it in `source`.  No header can be included: math builtins (exp, log1p, lgamma, ...)
 * are available without one.  `params` [n_params] (device, dtype; NULL exactly when n_params == 0) holds the
 * model's data and hyper-parameters and must outlive the handle.
 *
 * The source is compiled at run time by NVRTC (libnvrtc.so.12, loaded on first use) for sm_100a with
 * -std=c++17, plus --fmad=false in fp64 (the parity mode forbids contraction).  Compiled modules are cached for
 * the life of the process by (source, dims, dtype, prior/likelihood split) and never unloaded.  The handle works
 * everywhere a model handle does except the SMC, which needs the split (bk_model_create_cuda_prior_lik below):
 * HMCDiag, MALA and RW-Metropolis run one fused register-resident kernel per call for dims <= 32 (one thread per
 * chain; otherwise the generic engine), as do DrGhmcDiag and the Stretcher (see bk_drghmc_sample and
 * bk_stretch_move).  The fused kernels draw the same Philox words as every other engine; those of HMCDiag, MALA and
 * RW-Metropolis leave *cache_valid_host = 0.
 *
 * log_out [log_bytes] (may be NULL) receives NVRTC's log, truncated and NUL terminated; it includes ptxas's
 * register / spill report of every kernel.  Returns BK_E_INVALID on a bad argument or a compile error (the
 * first line of the log goes to bk_last_error), BK_E_UNSUPPORTED when NVRTC cannot be loaded, BK_E_CUDA when
 * the compiled module cannot be loaded (e.g. no device).  Arguments are checked before any device call. */
#define BK_USER_MAX_DIMS 65536
#define BK_USER_PRIOR_LIK_MAX_DIMS 256   /* bk_model_create_cuda_prior_lik */
BK_API int bk_model_create_cuda(const char* source, int64_t dims, int32_t dtype, const void* params,
                                int64_t n_params, uint64_t* handle_out, char* log_out, size_t log_bytes);

/* User-written model with a log_prior / log_likelihood split, for TemperedLikelihoodSMC: `source` defines the pair
 *
 *     __device__ bk_real log_prior_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
 *     __device__ bk_real log_likelihood_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
 *
 * each returning its log term and writing that term's gradient into grad[0 .. BK_DIMS).  The library derives
 * log_density_gradient = likelihood + prior (gradients likewise) after the source, so the handle (kind
 * BK_MODEL_USER_CUDA) also works everywhere a bk_model_create_cuda handle does.  In addition
 * bk_model_log_prior_likelihood accepts it, and the SMC entry points (bk_smc_move_weight, bk_smc_shard_move / _run,
 * ...) move its particles with one thread per particle: the same Philox words, resample indices, peer row reads and
 * mailbox messages as the built-in plugins, RW / MALA / HMC moves alike.  Same arguments, checks, log and return codes
 * as bk_model_create_cuda, with dims <= BK_USER_PRIOR_LIK_MAX_DIMS (the SMC's limit; each thread keeps a few
 * dims-element arrays). */
BK_API int bk_model_create_cuda_prior_lik(const char* source, int64_t dims, int32_t dtype, const void* params,
                                          int64_t n_params, uint64_t* handle_out, char* log_out, size_t log_bytes);

/* Initial states theta0 ~ N(0, I) (hmc.py:24-28, mala.py:26-30, metropolis.py:94-98; DrGhmcDiag's rho0,
 * drghmc.py:77): out [C, D] filled with device-Philox standard normals keyed by the GLOBAL chain id
 * (chain_offset + c) and draw index `draw` (the samplers reserve 0xFFFFFFFF for theta0 and 0xFFFFFFFE for
 * rho0), so the initial state of a chain does not depend on how the chains are sharded over GPUs. */
BK_API int bk_init_normal(void* out, int64_t C, int64_t D, int32_t dtype, uint64_t seed, uint64_t chain_offset,
                   uint32_t draw, void* stream);

/* ---- HMCDiag (hmc.py:9-63): n_draws calls of sample() for C chains ------- */
BK_API size_t bk_hmc_diag_workspace_bytes(uint64_t handle, int64_t C);
/* theta [C,D] in/out.  lp_cache [C] / grad_cache [C,D] hold log p and its
 * gradient at theta (in/out, only read when *cache_valid != 0; refreshed and
 * *cache_valid set to 1 on return; used by the GEMM-gradient models, ignored by
 * the fused separable kernels -- pass NULL there if you like).
 * metric: [D] or NULL (identity; the reference only supports None/size-1). */
BK_API int bk_hmc_diag_sample(uint64_t handle, void* theta, void* lp_cache, void* grad_cache,
                       int32_t* cache_valid_host, int64_t C, double stepsize, int32_t steps,
                       const void* metric, int64_t n_draws, const bk_rng* rng,
                       const bk_draw_out* out, void* ws, size_t ws_bytes, void* stream);

/* ---- MALA (mala.py:15-79) ----------------------------------------------- */
BK_API size_t bk_mala_workspace_bytes(uint64_t handle, int64_t C);
BK_API int bk_mala_sample(uint64_t handle, void* theta, void* lp_cache, void* grad_cache,
                   int32_t* cache_valid_host, int64_t C, double epsilon, int64_t n_draws,
                   const bk_rng* rng, const bk_draw_out* out, void* ws, size_t ws_bytes,
                   void* stream);

/* ---- Metropolis / MetropolisHastings with the built-in Gaussian random-walk
 * proposal theta' = theta + scale*z (metropolis.py:79-155; proposal family of
 * smc.py:79-89 / test_metropolis.py:114).  hastings != 0 also evaluates the
 * (cancelling) symmetric transition terms like MetropolisHastings does. ---- */
BK_API size_t bk_mh_rw_workspace_bytes(uint64_t handle, int64_t C);
BK_API int bk_mh_rw_sample(uint64_t handle, void* theta, void* lp_cache, int32_t* cache_valid_host,
                    int64_t C, double scale, int32_t hastings, int64_t n_draws,
                    const bk_rng* rng, const bk_draw_out* out, void* ws, size_t ws_bytes,
                    void* stream);

/* ---- Metropolis / MetropolisHastings with a user-written proposal (metropolis.py:79-135: proposal_fn and
 * transition_lp_fn written in CUDA C++).  `source` defines
 *
 *     __device__ void propose(const bk_real* theta, bk_real* proposal, const bk_real* z, const bk_real* u,
 *                             const bk_real* params);
 *     __device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* params);
 *
 * propose writes theta' into proposal[0 .. BK_DIMS) from z [BK_PROPOSAL_NORMALS] standard normals and u
 * [BK_PROPOSAL_UNIFORMS] uniforms in (0, 1) of this (chain, draw) -- the library draws all of them before every
 * call (streams: see bk_rng) -- and transition_log_density returns log q(to | from) up to a constant; it is required
 * only with has_transition = 1.  bk_real, BK_DIMS, the compile options, the absence of headers and the log are those
 * of bk_model_create_cuda; the source is compiled inside namespace bk_proposal, so its helpers may share names with a
 * model's.  BK_PROPOSAL_NORMALS = n_normals and BK_PROPOSAL_UNIFORMS = n_uniforms are compile-time constants.
 * `params` [n_params] (device, dtype; NULL exactly when n_params == 0) must outlive the handle.  Compiled programs
 * are cached for the life of the process and never unloaded.  Arguments are checked before any compilation or device
 * call: source and handle_out required, dims in [1, BK_USER_MAX_DIMS], n_normals in [0, BK_PROPOSAL_MAX_NORMALS],
 * n_uniforms in [0, BK_PROPOSAL_MAX_UNIFORMS].  Returns BK_E_INVALID on a bad argument or a compile error,
 * BK_E_UNSUPPORTED without NVRTC, BK_E_CUDA when the compiled module cannot be loaded.  Proposal handles have a
 * registry of their own: no model entry point accepts one. */
#define BK_PROPOSAL_MAX_NORMALS BK_USER_MAX_DIMS
#define BK_PROPOSAL_MAX_UNIFORMS 64
BK_API int bk_proposal_create_cuda(const char* source, int64_t dims, int32_t dtype, const void* params,
                                   int64_t n_params, int32_t n_normals, int32_t n_uniforms, int32_t has_transition,
                                   uint64_t* handle_out, char* log_out, size_t log_bytes);
BK_API int bk_proposal_destroy(uint64_t handle);
/* Engines: a user model (bk_model_create_cuda*) with dims <= 32 and a proposal with n_normals <= 32 run one fused
 * kernel per call (bk_user_mhp: one thread per chain, theta and log p(theta) in registers across the draws; leaves
 * *cache_valid_host = 0; compiled from the model's and the proposal's sources together, once per process, by
 * bk_mh_cuda_prepare or on the first call).  Every other model runs three launches per draw: the proposal
 * (bk_user_propose), the model's evaluation of the proposals and the accept test of bk_mh_rw_sample, with
 * lp_cache / cache_valid_host as there.  hastings != 0 adds transition_log_density(theta, theta') -
 * transition_log_density(theta', theta).  BK_E_INVALID when the model's and the proposal's dims or dtype differ,
 * when hastings != 0 and the proposal has no transition, or when INJECTED n_uniform != 1 + n_uniforms.  Draws are
 * [n_draws, C, D] only; streaming moments are folded from them. */
BK_API size_t bk_mh_cuda_workspace_bytes(uint64_t model, uint64_t proposal, int64_t C);
BK_API int bk_mh_cuda_prepare(uint64_t model, uint64_t proposal, char* log_out, size_t log_bytes);
BK_API int bk_mh_cuda_sample(uint64_t model, uint64_t proposal, void* theta, void* lp_cache,
                             int32_t* cache_valid_host, int64_t C, int32_t hastings, int64_t n_draws,
                             const bk_rng* rng, const bk_draw_out* out, void* ws, size_t ws_bytes, void* stream);

/* ---- DrGhmcDiag (drghmc.py:37-446) --------------------------------------
 * theta, rho [C,D] in/out; step_sizes_host[K], step_counts_host[K].
 * uniforms are consumed retry-test then accept-test per attempt
 * (drghmc.py:370,378): rng->n_uniform must be 2K in INJECTED mode.
 * Engines: iso / diagonal Gaussian plugins up to 256 dims run one fused kernel; a user model
 * (bk_model_create_cuda*) with dims <= 32 runs one fused kernel per call too (bk_user_drghmc: one
 * thread per chain, theta, rho, the gradient and log p(theta) in registers across the draws; compiled
 * from the model's source in a program of its own, once per process, by bk_drghmc_cuda_prepare or on
 * the first call); every other model runs the lockstep engine, with scratch from
 * bk_drghmc_workspace_bytes (0 on the fused engines). */
BK_API size_t bk_drghmc_workspace_bytes(uint64_t handle, int64_t C, int32_t max_proposals);
/* Compiles and loads the fused DrGHMC program of a user model that takes that engine, so that the first
 * bk_drghmc_sample does not pay the NVRTC compile; log_out as bk_model_create_cuda's (ptxas's report of
 * bk_user_drghmc).  BK_OK with an empty log for any other model, BK_E_HANDLE for an unknown handle,
 * BK_E_INVALID on a compile error (with the log), BK_E_UNSUPPORTED without NVRTC. */
BK_API int bk_drghmc_cuda_prepare(uint64_t handle, char* log_out, size_t log_bytes);
BK_API int bk_drghmc_sample(uint64_t handle, void* theta, void* rho, int64_t C, int32_t max_proposals,
                     const double* step_sizes_host, const int32_t* step_counts_host,
                     double damping, int32_t prob_retry, const void* metric, int64_t n_draws,
                     const bk_rng* rng, const bk_draw_out* out, int32_t* n_uniform_used_out,
                     void* ws, size_t ws_bytes, void* stream);

/* ---- TemperedLikelihoodSMC (smc.py:12-89) -------------------------------- */
/* One temperature step n (1-based) of T for M particles, RW-Metropolis kernel
 * of smc.py:79-89 targeting time(n-1) (smc.py:54-57) fused with the importance
 * log-weights lp_n - lp_{n-1} of smc.py:67-70.  thetas [M,D] in/out;
 * logw_out [M].  rng: normals [1,M,D], uniforms [1,M,1] when INJECTED;
 * draw_offset = n. */
BK_API int bk_smc_move_weight(uint64_t handle, void* thetas, int64_t M, int32_t n, int32_t T,
                       double scale, const bk_rng* rng, void* logw_out, int32_t* accept_out,
                       void* stream);
/* Same move with the previous temperature's resampling gather folded into the
 * read: particle m starts from src[src_idx[m]] (src_idx NULL: src[m]) and the
 * moved particle is written to thetas[m] -- thetas[idxs] (smc.py:75) followed by
 * the kernel loop (smc.py:54-57) in one pass over HBM.  src [*, D] is the
 * (all-gathered) particle array the indices refer to; src != thetas when
 * src_idx is given. */
BK_API int bk_smc_gather_move_weight(uint64_t handle, const void* src, const int64_t* src_idx,
                       void* thetas, int64_t M, int32_t n, int32_t T, double scale,
                       const bk_rng* rng, void* logw_out, int32_t* accept_out, void* stream);
/* ... and with log-weights carried over from temperatures that did not resample
 * (adaptive resampling): logw_out[m] = logw_prev[m] + (lp_n - lp_{n-1}); logw_prev
 * NULL = the call above. */
BK_API int bk_smc_gather_move_weight_acc(uint64_t handle, const void* src, const int64_t* src_idx,
                       void* thetas, int64_t M, int32_t n, int32_t T, double scale,
                       const bk_rng* rng, const void* logw_prev, void* logw_out,
                       int32_t* accept_out, void* stream);
/* Adaptive resampling (SURVEY 8f-4; the reference resamples unconditionally,
 * smc.py:60): after bk_smc_weight_stats and bk_smc_resample_indices, keep the
 * computed indices and zero the log-weights iff (sum w)^2 / sum w^2 <
 * ess_threshold, else overwrite idx with the identity (point_offset + i) and keep
 * the accumulated log-weights.  Decided on device from `stats`; *resampled_out
 * (device int32, may be NULL) records the decision. */
BK_API int bk_smc_adaptive_select(const double* stats, double ess_threshold, int64_t n_points,
                       int64_t point_offset, int64_t* idx_inout, void* logw_inout, int32_t dtype,
                       int32_t* resampled_out, void* stream);
BK_API size_t bk_smc_resample_workspace_bytes(int64_t M);
/* local reduction of the log-weights: stats_out[0] = max, [1] = sum exp(logw -
 * shift), [2] = sum exp(..)^2 where shift = max (SYSTEMATIC) or 0
 * (MULTINOMIAL, the reference does not shift: smc.py:67); always fp64.  The
 * multi-GPU path all-reduces these between this call and bk_smc_resample. */
BK_API int bk_smc_weight_stats(const void* logw, int64_t M, int32_t dtype, int32_t mode,
                        double* stats_out, void* ws, size_t ws_bytes, void* stream);
/* indices of importance_resample (smc.py:64-75) for M weights (multi-GPU:
 * the all-gathered log-weights, so every rank builds the same CDF):
 *   p_i = exp(logw_i - shift) / total;  cdf = cumsum(p);  cdf /= cdf[-1]
 * MULTINOMIAL: idx_i = searchsorted(cdf, u_i, 'right') (== legacy
 * np.random.choice, SURVEY.md 2.1-9) with u [n_points] INJECTED via
 * `uniforms`, else Philox keyed by the global point index.  SYSTEMATIC:
 * points (point_offset + i + u0) / M with u0 = uniforms[0] or Philox; pass
 * total = 1 (the CDF is normalised by its last entry).  This call resolves
 * the n_points points starting at global point index point_offset (a rank's
 * slice).  idx_out [n_points] int64; cdf_out [M] f64 or NULL (scratch in ws). */
BK_API int bk_smc_resample_indices(const void* logw, int64_t M, int32_t dtype, int32_t mode,
                            double shift, double total, const void* uniforms, const bk_rng* rng,
                            int64_t n_points, int64_t point_offset, int64_t* idx_out,
                            void* cdf_out, void* ws, size_t ws_bytes, void* stream);
/* Same, with the normaliser read ON DEVICE from `stats` (the 3 doubles
 * bk_smc_weight_stats wrote): no host round trip between the two calls. */
BK_API int bk_smc_resample_indices_dev(const void* logw, int64_t M, int32_t dtype, int32_t mode,
                            const double* stats, const void* uniforms, const bk_rng* rng,
                            int64_t n_points, int64_t point_offset, int64_t* idx_out,
                            void* cdf_out, void* ws, size_t ws_bytes, void* stream);
/* thetas[idxs] (smc.py:75): out [M,D] = src[idx] */
BK_API int bk_gather_rows(const void* src, const int64_t* idx, int64_t M, int64_t D, int32_t dtype,
                   void* out, void* stream);

/* ---- TemperedLikelihoodSMC sharded over G GPUs (SURVEY 8(e), north_star item 4) ----------------
 * One process per GPU; rank r owns the contiguous particle range
 *   lo(r) = r * (M / G) + min(r, M % G),  n(r) = M / G + (r < M % G).
 * Per temperature the ranks exchange NO particle array and call NO host-side collective: the arrays
 * below are PEER-ACCESSIBLE device memory (NVLink P2P / torch symmetric memory; with world == 1 plain
 * device memory) and the kernels talk through them --
 *   max message   (end of the move kernel)    local max of the log-weights            16 B per peer
 *   mass message  (end of the scan kernel)    local fixed-point weight mass, sum w^2  32 B per peer
 *   indices       (resolve kernel)            global particle id of every offspring,   8 B per slot
 *                                             stored into the slot owner's idx array
 *   done message  (end of the resolve kernel)                                          8 B per peer
 *   particle rows (next move kernel)          row idx[m] read from its owner's array   D * s per row
 * SYSTEMATIC resampling is defined in exact integer arithmetic so that the indices do not depend on
 * G:  w_i = rint(exp(logw_i - max) * 2^s),  s = 61 - ceil(log2 M);  C = cumsum(w) (int64, exact);
 * point k has threshold t_k = floor((k + u0) * (W / M)) (fp64 ops in this order, W = sum w, clamped to
 * W - 1) and selects the first particle with C > t_k.  Rank r resolves exactly the points whose
 * threshold falls into its own interval [O_r, O_r + W_r).  MULTINOMIAL (the reference's
 * np.random.choice, smc.py:64-75) keeps its fp64 CDF: every rank reads all log-weights from its
 * peers (M * s bytes) and resolves its own slots against the full CDF -- bit-identical to one GPU.
 * All buffers are caller-owned; `ws` (bk_smc_shard_workspace_bytes) and the mailboxes must be zeroed
 * ONCE before the first step.  A wait that is not satisfied within 20 s (dead peer) sets mailbox word
 * 0 to 1 and the kernels finish on garbage instead of hanging; 2 = every weight vanished. */
/* the Markov kernel that moves a particle at temperature time(n-1) (smc.py:54-57):
 *   RW        theta* = theta + scale z, Metropolis test                       (metropolis_kernel, smc.py:79-89)
 *   MALA      one Langevin proposal with step `scale` on the tempered density (mala.py:40-66; smc.py:78 TODO)
 *   HMC       `steps` leapfrog steps of size `scale`, identity metric          (hmc.py:40-63;  smc.py:78 TODO)
 *   PROPOSAL  theta* = propose(theta, z, u) of the user proposal `proposal` (bk_proposal_create_cuda), then the
 *             Metropolis test on the tempered density plus, when the proposal was created with has_transition,
 *             the Hastings term transition_log_density(theta, theta*) - transition_log_density(theta*, theta)
 *             (smc.py:54-57 with any kernel).  User prior/likelihood models only (bk_model_create_cuda_prior_lik;
 *             restate GAUSS_PRIOR_LIK / BINOMIAL_LOGIT as one): BK_E_UNSUPPORTED otherwise.  The proposal's dims
 *             and dtype must be the model's and n_normals <= BK_SMC_PROPOSAL_MAX_NORMALS; INJECTED streams need
 *             n_uniform = 1 + n_uniforms (layout: the note after bk_rng).  `scale` and `steps` are not read.
 * `proposal` is read only by the PROPOSAL kind: initialisers such as {BK_SMC_KERNEL_RW, 0, scale} leave it 0. */
enum { BK_SMC_KERNEL_RW = 0, BK_SMC_KERNEL_MALA = 1, BK_SMC_KERNEL_HMC = 2, BK_SMC_KERNEL_PROPOSAL = 3 };
typedef struct bk_smc_kernel { int32_t kind; int32_t steps; double scale; uint64_t proposal; } bk_smc_kernel;
/* one thread per particle keeps the proposal's normals in local memory: the bound keeps that array small */
#define BK_SMC_PROPOSAL_MAX_NORMALS 512
/* Checks (model, proposal) as bk_smc_shard_move does for the PROPOSAL kind and compiles their fused program
 * (bk_user_smc_mhp; once per process and pair, shared with bk_mh_cuda_prepare), so that the first move does not
 * pay the NVRTC compile.  log_out as bk_model_create_cuda's.  BK_E_HANDLE for an unknown handle, BK_E_INVALID
 * on a bad argument or a compile error (with the log), BK_E_UNSUPPORTED for a model the proposal move does not
 * serve. */
BK_API int bk_smc_cuda_prepare(uint64_t model, uint64_t proposal, char* log_out, size_t log_bytes);
#define BK_SMC_MAX_WORLD 16
#define BK_SMC_MAILBOX_BYTES 4096
typedef struct bk_smc_shard {
    int32_t  rank, world;
    int64_t  M;                                   /* GLOBAL particle count                           */
    uint64_t epoch;                               /* number of this temperature step: 1, 2, ... (the
                                                     same on every rank)                             */
    void*    particles[2][BK_SMC_MAX_WORLD];      /* every rank's two particle arrays [n(r), D]:
                                                     step e writes [e & 1], reads [(e - 1) & 1]      */
    void*    llpr[2][BK_SMC_MAX_WORLD];           /* every rank's (log_likelihood, log_prior) pairs
                                                     [n(r), 2] of the particles in the same-numbered
                                                     particle array: a move starts from its parent's
                                                     pair instead of re-evaluating the model         */
    void*    logw[BK_SMC_MAX_WORLD];              /* every rank's log-weights [n(r)]                 */
    int64_t* idx[BK_SMC_MAX_WORLD];               /* every rank's resample indices [n(r)], global ids */
    void*    mailbox[BK_SMC_MAX_WORLD];           /* every rank's mailbox (BK_SMC_MAILBOX_BYTES)      */
} bk_smc_shard;
BK_API size_t bk_smc_shard_workspace_bytes(int64_t M, int32_t world, int32_t mode);
/* Move + weight of step n (smc.py:54-57, 67-70) for this rank's particles; the local max of the
 * log-weights is posted to every rank from the kernel's last CTA.  Particle m starts from
 * src_local[m] when src_local != NULL (first step, or after the caller replaced the particles),
 * else from row idx[m] of the step-(epoch-1) arrays (peer reads) -- after waiting, in the kernel, for
 * every rank's done message of step epoch-1.  accumulate != 0: logw += (adaptive resampling).
 * rng->chain_offset must be lo(rank). */
BK_API int bk_smc_shard_move(uint64_t handle, const bk_smc_shard* sh, const void* src_local, int32_t n,
                      int32_t T, const bk_smc_kernel* kernel, const bk_rng* rng, int32_t accumulate,
                      int32_t* accept_out, void* ws, size_t ws_bytes, void* stream);
/* Normaliser + resampling of step `epoch`.  SYSTEMATIC: two kernels (fixed-point scan; resolve).
 * uniforms: the injected u0 [1] (SYSTEMATIC) or this rank's [n(rank)] uniforms (MULTINOMIAL), or NULL
 * (Philox: rng).  ess_threshold > 0 (SYSTEMATIC only): resample iff (sum w)^2 / sum w^2 <
 * ess_threshold, else identity indices and the log-weights are kept (decided on device, identically
 * on every rank).  stats_out (device, 4 doubles, may be NULL): max, sum exp(logw - max), sum exp(..)^2,
 * resampled (0/1).  phase: 0 = everything; 1 / 2 = first / second kernel only (a single-GPU
 * "fake world" test drives G ranks in lockstep on one device). */
BK_API int bk_smc_shard_resample(const bk_smc_shard* sh, int32_t dtype, int32_t mode, const void* uniforms,
                          const bk_rng* rng, double ess_threshold, int32_t phase, double* stats_out,
                          void* ws, size_t ws_bytes, void* stream);
/* run() (smc.py:39-41) for temperatures n_from..n_to in ONE call: move + resample of every step enqueued
 * back to back from C (3 launches per temperature, no per-step host work -- at 8 GPUs a temperature of c4 is
 * ~60 us of device time, less than two Python-level calls cost).  sh->epoch is the epoch of step n_from and
 * advances by one per step (the caller continues with epoch + n_to - n_from + 1); Philox only (rng->mode),
 * rng->draw_offset is ignored: step n draws with draw_offset = n, like the step-wise calls.
 * stats_out: [n_to - n_from + 1, 4] doubles or NULL; accept_out: flags of the LAST step or NULL. */
BK_API int bk_smc_shard_run(uint64_t handle, const bk_smc_shard* sh, const void* src_local, int32_t n_from,
                     int32_t n_to, int32_t T, const bk_smc_kernel* kernel, const bk_rng* rng, int32_t mode,
                     double ess_threshold, double* stats_out, int32_t* accept_out, void* ws, size_t ws_bytes,
                     void* stream);
/* thetas[idxs] (smc.py:75) materialised: out [n(rank), D] = rows idx[m] of the step-`epoch` arrays. */
BK_API int bk_smc_shard_gather(const bk_smc_shard* sh, int64_t D, int32_t dtype, void* out, void* stream);

/* ---- Stretcher: affine-invariant ensemble sampler (ensemble.py:9-66, the
 * Goodman & Weare stretch move sketched in the reference's comments) --------
 * One call moves the n_active walkers `active` [n_active, D] (in/out, with
 * their cached log densities lp_active; *lp_valid_host = 0 re-evaluates them)
 * against the complementary half `other` [n_other, D]:
 *   j = floor(u0 * n_other);  z = (1/sqrt(a) + (sqrt(a) - 1/sqrt(a)) u1)^2
 *   theta* = other[j] + z (theta_k - other[j])
 *   accept iff log(u2) < (D - 1) log z + log p(theta*) - log p(theta_k)
 * u0..u2: Philox keyed by (seed, chain_offset + k, draw_offset) or INJECTED
 * uniforms [n_active, 3].  accept_out [n_active] or NULL.
 * Engines: a user model (bk_model_create_cuda*) with dims <= 32 runs one fused kernel per call
 * (bk_user_stretch: one thread per walker, the proposal in registers, lp_active kept as on the
 * other engine; compiled from the model's source in a program of its own, once per process, by
 * bk_stretch_cuda_prepare or on the first call); every other model runs three launches (propose,
 * the model's density, accept) with scratch from bk_stretch_workspace_bytes (0 on the fused engine). */
BK_API size_t bk_stretch_workspace_bytes(uint64_t handle, int64_t n_active);
/* Compiles and loads the fused Stretcher program of a user model that takes that engine, so that the
 * first bk_stretch_move does not pay the NVRTC compile; log_out as bk_model_create_cuda's (ptxas's
 * report of bk_user_stretch).  BK_OK with an empty log for any other model, BK_E_HANDLE for an
 * unknown handle, BK_E_INVALID on a compile error (with the log), BK_E_UNSUPPORTED without NVRTC. */
BK_API int bk_stretch_cuda_prepare(uint64_t handle, char* log_out, size_t log_bytes);
BK_API int bk_stretch_move(uint64_t handle, void* active, void* lp_active, int32_t* lp_valid_host,
                    const void* other, int64_t n_active, int64_t n_other, double a,
                    const bk_rng* rng, int32_t* accept_out, void* ws, size_t ws_bytes, void* stream);

/* ---- diagnostics -------------------------------------------------------- */
/* Where the draws of series s live: element t of series s is
 *   x[(s / n_inner) * outer_stride + (s % n_inner) * inner_stride + t * draw_stride]
 * (strides in elements), so [chains, draws], [chains, draws, params] and the
 * samplers' own [draws, chains, params] output are all consumed in place. */
typedef struct bk_series_layout {
    int64_t n_series, n_draws, n_inner, outer_stride, inner_stride, draw_stride;
} bk_series_layout;

/* Rank normalisation of ONE parameter (rhat.py:27-108): the layout's series are
 * that parameter's chains (n_series chains x n_draws draws each); ranks are taken
 * over the concatenation of the chains in series order (np.concatenate,
 * rhat.py:51), ascending from 1, ties in flattened order (stable; the reference's
 * tie order is implementation defined).  ranks_out / z_out [n_series * n_draws]
 * f64 in that same flattened order (either may be NULL):
 *   z = Phi^-1((rank - 0.325) / (S - 0.25)),  S = n_series * n_draws   (rhat.py:106)
 * Hand-written stable LSD radix sort + normcdfinv; S < 2^32. */
BK_API size_t bk_rank_normalize_workspace_bytes(int64_t n_total, int32_t dtype);
BK_API int bk_rank_normalize(const void* x, int32_t dtype, const bk_series_layout* layout,
                      double* ranks_out, double* z_out, void* ws, size_t ws_bytes, void* stream);

BK_API size_t bk_autocorr_workspace_bytes(int64_t n_series, int64_t N);
/* autocorr.py:6-33 -- all N lags of the biased estimator, fp64 accumulate;
 * out [n_series, N] f64 */
BK_API int bk_autocorr(const void* x, int32_t dtype, const bk_series_layout* layout, double* out,
                       void* ws, size_t ws_bytes, void* stream);
/* Scratch for bk_iat_ess: 0 when every series' draws are contiguous; otherwise room to gather
 * blocks of up to 65,536 series into [series, draws] form (optional: without it the strided
 * series are read in place, correct but sector-inefficient). */
BK_API size_t bk_iat_ess_workspace_bytes(int32_t dtype, const bk_series_layout* layout);
/* iat_ipse/iat_imse (iat.py:46-135) and ess_* (ess.py:5-69); outputs [n_series] f64 */
BK_API int bk_iat_ess(const void* x, int32_t dtype, const bk_series_layout* layout, int32_t estimator,
                      double* iat_out, double* ess_out, void* ws, size_t ws_bytes, void* stream);
/* per-series mean and ddof=1 variance (rhat.py:165-166); outputs [n_series] f64 */
BK_API int bk_chain_moments(const void* x, int32_t dtype, const bk_series_layout* layout,
                            double* mean_out, double* var_out, void* stream);
/* Streaming moments: fold a batch of draws [n_draws, n_elems] (the samplers'
 * [n, C, D] output, n_elems = C * D) into running per-element mean / M2 (sum of
 * squared deviations) that already cover n0 draws (n0 = 0 initialises them).
 * var(ddof=1) = M2 / (n0 + n_draws - 1): R-hat (rhat.py:165-170) then needs no
 * pass over the stored chains -- bk_rhat_from_moments on the result. */
BK_API int bk_moments_accumulate(const void* draws, int32_t dtype, int64_t n_draws, int64_t n_elems,
                          int64_t n0, double* mean_inout, double* m2_inout, void* stream);
/* rhat (rhat.py:111-171) from per-chain moments laid out [n_chains, n_params];
 * lengths [n_chains] (ragged allowed) or NULL with common length N.
 * out [n_params] f64 */
BK_API int bk_rhat_from_moments(const double* mean, const double* var, const int64_t* lengths,
                                int64_t N, int64_t n_chains, int64_t n_params, double* out,
                                void* stream);

/* Cross-rank R-hat (rhat.py:163-170) when the chains are sharded over GPUs: instead of gathering
 * per-chain moments, every rank reduces its own chains to per-parameter sums which are all-reduced
 * (SUM) -- 4 doubles per parameter on the wire in total.  Two passes keep var(chain means) free of
 * cancellation:
 *   pass 1 (ref = NULL): sums [n_params, 3] = {n_chains, sum mean, sum var};  all-reduce;
 *                        bk_rhat_from_sums(sums, NULL, .., ref_out, NULL) -> grand means [n_params]
 *   pass 2 (ref = grand means): sqdev [n_params] = sum (mean - ref)^2;        all-reduce;
 *                        bk_rhat_from_sums(sums, sqdev, .., NULL, out)    -> R-hat [n_params]
 * for the common chain length N (NaN with fewer than two chains in total).  mean / var
 * [n_chains, n_params] as written by bk_chain_moments. */
BK_API int bk_rhat_partial_sums(const double* mean, const double* var, int64_t n_chains, int64_t n_params,
                         const double* ref, double* out, void* stream);
BK_API int bk_rhat_from_sums(const double* sums, const double* sqdev, int64_t n_params, int64_t N,
                      double* ref_out, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BK_B200_H */
