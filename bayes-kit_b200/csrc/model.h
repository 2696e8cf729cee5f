// Model plugin registry (host side) and batched device evaluation.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace bk {

struct Model {
    bk_model_desc d;
    // derived operands living in the caller-provided model workspace
    void* Pmu = nullptr;            // [D]  P * mu (DENSE with mu), dtype
    __nv_bfloat16* P_hi = nullptr;  // [Dp, Dp] bf16(P), zero padded   (fp32 DENSE: tcgen05 operand)
    __nv_bfloat16* P_lo = nullptr;  // [Dp, Dp] bf16(P - P_hi)
    int64_t Dp = 0;                 // D rounded up to 128
    __nv_bfloat16* Xb = nullptr;    // [Np, 128] bf16(X), zero padded      (fp32 HIER_LOGREG: tcgen05 operands)
    __nv_bfloat16* Xlo = nullptr;   // [Np, 128] bf16(X - Xb): split-precision logits
    float* yp = nullptr;            // [Np] responses, zero padded
    float* yh = nullptr;            // [Np] responses - 1/2 (0 on padded rows)
    const struct Program* user = nullptr;   // USER_CUDA: the model's runtime-compiled program (user_model.cu)
    const void* user_params = nullptr;      // USER_CUDA: [n_params] caller array, dtype
    bool separable() const {
        return d.kind == BK_MODEL_ISO_GAUSS || d.kind == BK_MODEL_DIAG_GAUSS;
    }
};

// returns nullptr (and sets the error) for an unknown handle
const Model* get_model(uint64_t handle);
// adds m to the registry
int register_model(const Model& m, uint64_t* handle_out);

// user-written CUDA models (user_model.cu).  The fused register-resident samplers serve D <= USER_FUSED_MAX_D: up to
// there both measured models gain more than 10x over the generic engine (DESIGN.md 4.4a).  Defining
// BK_USER_FUSED_MAX_D at build time moves the threshold (scripts/time_user_model.py measures beyond it that way).
#ifndef BK_USER_FUSED_MAX_D
#define BK_USER_FUSED_MAX_D 32
#endif
constexpr int USER_FUSED_MAX_D = BK_USER_FUSED_MAX_D;
struct UserRunArgs;
struct UserSmcArgs;
struct UserProposeArgs;
// user-written CUDA proposals (bk_proposal_create_cuda)
struct UserProposal {
    const struct Program* lib;   // the proposal's own program (bk_user_propose)
    int64_t dims;
    int32_t dtype, n_normals, n_uniforms, has_transition;
    const void* params;          // [n_params] caller array, dtype, or NULL
};
// returns nullptr (and sets the error) for an unknown handle
const UserProposal* get_proposal(uint64_t handle);

int user_eval(const Model& m, const void* theta, int64_t C, void* lp, void* grad, void* ws, size_t ws_bytes,
              cudaStream_t st);
bool user_fused(const Model& m);
// theta, the model's params, the streams and the outputs of a fused launch; the caller sets the sampler's fields
UserRunArgs user_args(const Model& m, void* theta, int64_t C, int64_t n, const bk_rng* rng, const bk_draw_out& out);
// bk_user_hmc / mala / mh (algo: ALGO_*), or with a proposal p bk_user_mhp of the program of (m, p)
int user_fused_sample(const Model& m, const UserProposal* p, int algo, const UserRunArgs& a, int32_t* cache_valid,
                      cudaStream_t st);
// prior/likelihood user models (bk_model_create_cuda_prior_lik): log_prior / log_likelihood of theta [C, D] (each
// output nullable) and TemperedLikelihoodSMC's move + weight kernel (move: BK_SMC_KERNEL_*; the PROPOSAL move runs
// bk_user_smc_mhp of the program of (m, p))
bool user_prior_lik(const Model& m);
int user_log_prior_likelihood(const Model& m, const void* theta, int64_t C, void* lprior, void* llik, cudaStream_t st);
int user_smc_move(const Model& m, const UserProposal* p, int move, const UserSmcArgs& a, cudaStream_t st);
// the fused bk_user_mhp serves (m, p): a user model with dims <= USER_FUSED_MAX_D and n_normals <= USER_FUSED_MAX_D
bool user_mhp_fusable(const Model& m, const UserProposal& p);
// The programs of (m, p) and of m's DrGHMC kernel are compiled (once per process) by these or on their first launch;
// log_out as bk_model_create_cuda's, `who` names the caller in errors.  K <= DR_KMAX (drghmc.cu).
int user_mhp_prepare(const Model& m, const UserProposal& p, const char* who, char* log_out, size_t log_bytes);
int user_drghmc_prepare(const Model& m, char* log_out, size_t log_bytes);
int user_drghmc_sample(const Model& m, void* theta, void* rho, int64_t C, int K, const double* sizes,
                       const int32_t* counts, double damping, int prob_retry, const void* metric, int64_t n,
                       const bk_rng* rng, const bk_draw_out& out, int32_t* n_used, cudaStream_t st);
// The Stretcher on a user model with dims <= USER_FUSED_MAX_D: the program of bk_user_stretch, compiled (once per
// process) by the prepare or on the first move, and one half-step of bk_stretch_move in one launch.  eval_lp: lp [n]
// is not valid and the kernel evaluates it first.
int user_stretch_prepare(const Model& m, char* log_out, size_t log_bytes);
int user_stretch_move(const Model& m, void* active, void* lp, bool eval_lp, const void* other, int64_t n, int64_t mo,
                      double a, const bk_rng* rng, int32_t* accept, cudaStream_t st);
// three-launch path: Philox scratch of bk_user_propose ([C, n_normals] and [C, n_uniforms]) and its launch
size_t user_propose_ws_bytes(const UserProposal& p, int64_t C);
int user_propose(const UserProposal& p, const UserProposeArgs& a, cudaStream_t st);

size_t model_eval_ws_bytes(const Model& m, int64_t C);
// true when model_eval(..., precise=false) is a genuinely cheaper (tensor-core) evaluation
bool model_has_fast_path(const Model& m);
// theta [C,D] -> lp [C], grad [C,D] (nullable).  All on `st`.  precise = false lets a plugin
// answer with its reduced-precision tensor-core path: allowed for INTERIOR leapfrog
// gradients only (any deterministic gradient keeps the leapfrog map reversible and
// volume preserving); everything that enters a Metropolis test must be precise.
int model_eval(const Model& m, const void* theta, int64_t C, void* lp, void* grad, void* ws,
               size_t ws_bytes, cudaStream_t st, bool precise = true);

// hierarchical logistic regression evaluator (logreg.cu)
size_t hlr_eval_ws_bytes(const Model& m, int64_t C);
int hlr_eval(const Model& m, const void* theta, int64_t C, void* lp, void* grad, void* ws, size_t ws_bytes,
             cudaStream_t st, bool precise);
// tcgen05 path (logreg_tc.cu)
size_t hlr_tc_model_ws_bytes(const bk_model_desc& d);
int hlr_tc_prepare(Model& m, void* ws, size_t ws_bytes, cudaStream_t st);
bool hlr_tc_enabled(const Model& m);
size_t hlr_tc_eval_ws_bytes(const Model& m, int64_t C);
enum { HLR_TC_GRAD = 0, HLR_TC_GRAD_LL = 1, HLR_TC_LP = 2 };
int hlr_tc_partial(const Model& m, const float* theta, int64_t C, void* ws, size_t ws_bytes, float** part_g,
                   float** part_ll, int* n_split, cudaStream_t st, int mode, bool operand_ready = false,
                   __nv_bfloat16** operand = nullptr);
// interior leapfrog step of HMC on this plugin: tensor-core gradient of q, then ONE kernel that finishes
// the gradient, applies kick + drift to (r, q) in place and writes the next launch's bf16 operand.
// operand_ready: the operand of q was written by the previous call (same ws, same C).
int hlr_tc_interior_step(const Model& m, float* q, float* r, int64_t C, float eps, const float* metric,
                         bool operand_ready, void* ws, size_t ws_bytes, cudaStream_t st);
// n_steps of them; one persistent launch when the grid fits the device in one wave (logreg_tc.cu)
int hlr_tc_interior_steps(const Model& m, float* q, float* r, int64_t C, float eps, const float* metric, int n_steps,
                          void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace bk
