"""ctypes binding of libbk_b200.so (the C ABI declared in include/bk.h).

There is no CPU fallback: if the CUDA library is missing or does not load,
importing the samplers fails loudly here.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BK_LIB") or os.path.join(_HERE, "libbk_b200.so")   # BK_LIB: experiment builds (scripts/build_variant.sh)

BK_OK, BK_E_INVALID, BK_E_UNSUPPORTED, BK_E_CUDA, BK_E_WORKSPACE, BK_E_HANDLE = 0, -1, -2, -3, -4, -5
BK_F32, BK_F64 = 0, 1
MODEL_ISO, MODEL_DIAG, MODEL_DENSE, MODEL_HLR, MODEL_GPL, MODEL_BINOM, MODEL_USER = range(7)
SMC_KERNEL_RW, SMC_KERNEL_MALA, SMC_KERNEL_HMC, SMC_KERNEL_PROPOSAL = 0, 1, 2, 3
SMC_PROPOSAL_MAX_NORMALS = 512
SMC_MAX_WORLD, SMC_MAILBOX_BYTES = 16, 4096
RNG_PHILOX, RNG_INJECTED = 0, 1
RESAMPLE_MULTINOMIAL, RESAMPLE_SYSTEMATIC = 0, 1
IAT_IPSE, IAT_IMSE = 0, 1
PROF_GRAD, PROF_SAMPLER, PROF_STEP = 0, 1, 2

vp, i32, i64, u64, f64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double, C.c_size_t


class ModelDesc(C.Structure):
    _fields_ = [("kind", i32), ("dtype", i32), ("dims", i64), ("sigma", f64), ("mu", vp),
                ("prec", vp), ("P", vp), ("m0", vp), ("p0", vp), ("X", vp), ("y", vp),
                ("n_obs", i64), ("scalars", f64 * 8)]


class Rng(C.Structure):
    _fields_ = [("mode", i32), ("n_uniform", i32), ("seed", u64), ("draw_offset", u64),
                ("chain_offset", u64), ("normals", vp), ("uniforms", vp)]


class SmcKernel(C.Structure):
    _fields_ = [("kind", i32), ("steps", i32), ("scale", f64), ("proposal", u64)]


class SmcShard(C.Structure):
    _fields_ = [("rank", i32), ("world", i32), ("M", i64), ("epoch", u64),
                ("particles", (vp * SMC_MAX_WORLD) * 2), ("llpr", (vp * SMC_MAX_WORLD) * 2), ("logw", vp * SMC_MAX_WORLD),
                ("idx", vp * SMC_MAX_WORLD), ("mailbox", vp * SMC_MAX_WORLD)]


class DrawOut(C.Structure):
    _fields_ = [("draws", vp), ("logp", vp), ("accept", vp), ("layout", i32), ("mom_mean", vp), ("mom_m2", vp),
                ("mom_n0", i64)]


DRAWS_NCD, DRAWS_CDN = 0, 1


class SeriesLayout(C.Structure):
    _fields_ = [("n_series", i64), ("n_draws", i64), ("n_inner", i64), ("outer_stride", i64),
                ("inner_stride", i64), ("draw_stride", i64)]


class BkError(RuntimeError):
    pass


_SIGNATURES = {
    "bk_last_error": (C.c_char_p, []),
    "bk_abi_version": (C.c_int, []),
    "bk_launch_count": (u64, []),
    "bk_profile_enable": (C.c_int, [i32]),
    "bk_profile_read": (C.c_int, [i32, C.POINTER(f64), C.POINTER(u64)]),
    "bk_model_workspace_bytes": (sz, [C.POINTER(ModelDesc)]),
    "bk_model_create": (C.c_int, [C.POINTER(ModelDesc), vp, sz, vp, C.POINTER(u64)]),
    "bk_model_destroy": (C.c_int, [u64]),
    "bk_model_dims": (i64, [u64]),
    "bk_model_eval_workspace_bytes": (sz, [u64, i64]),
    "bk_model_log_density_gradient": (C.c_int, [u64, vp, i64, vp, vp, vp, sz, vp]),
    "bk_model_log_density_gradient_fast": (C.c_int, [u64, vp, i64, vp, vp, vp, sz, vp]),
    "bk_model_log_prior_likelihood": (C.c_int, [u64, vp, i64, vp, vp, vp]),
    "bk_model_create_cuda": (C.c_int, [C.c_char_p, i64, i32, vp, i64, C.POINTER(u64), C.c_char_p, sz]),
    "bk_model_create_cuda_prior_lik": (C.c_int, [C.c_char_p, i64, i32, vp, i64, C.POINTER(u64), C.c_char_p, sz]),
    "bk_proposal_create_cuda": (C.c_int, [C.c_char_p, i64, i32, vp, i64, i32, i32, i32, C.POINTER(u64), C.c_char_p,
                                          sz]),
    "bk_proposal_destroy": (C.c_int, [u64]),
    "bk_mh_cuda_workspace_bytes": (sz, [u64, u64, i64]),
    "bk_mh_cuda_prepare": (C.c_int, [u64, u64, C.c_char_p, sz]),
    "bk_mh_cuda_sample": (C.c_int, [u64, u64, vp, vp, C.POINTER(i32), i64, i32, i64, C.POINTER(Rng), C.POINTER(DrawOut),
                                    vp, sz, vp]),
    "bk_init_normal": (C.c_int, [vp, i64, i64, i32, u64, u64, C.c_uint32, vp]),
    "bk_hmc_diag_workspace_bytes": (sz, [u64, i64]),
    "bk_hmc_diag_sample": (C.c_int, [u64, vp, vp, vp, C.POINTER(i32), i64, f64, i32, vp, i64,
                                     C.POINTER(Rng), C.POINTER(DrawOut), vp, sz, vp]),
    "bk_mala_workspace_bytes": (sz, [u64, i64]),
    "bk_mala_sample": (C.c_int, [u64, vp, vp, vp, C.POINTER(i32), i64, f64, i64, C.POINTER(Rng),
                                 C.POINTER(DrawOut), vp, sz, vp]),
    "bk_mh_rw_workspace_bytes": (sz, [u64, i64]),
    "bk_mh_rw_sample": (C.c_int, [u64, vp, vp, C.POINTER(i32), i64, f64, i32, i64, C.POINTER(Rng),
                                  C.POINTER(DrawOut), vp, sz, vp]),
    "bk_drghmc_workspace_bytes": (sz, [u64, i64, i32]),
    "bk_drghmc_cuda_prepare": (C.c_int, [u64, C.c_char_p, sz]),
    "bk_drghmc_sample": (C.c_int, [u64, vp, vp, i64, i32, C.POINTER(f64), C.POINTER(i32), f64, i32,
                                   vp, i64, C.POINTER(Rng), C.POINTER(DrawOut), vp, vp, sz, vp]),
    "bk_stretch_workspace_bytes": (sz, [u64, i64]),
    "bk_stretch_cuda_prepare": (C.c_int, [u64, C.c_char_p, sz]),
    "bk_stretch_move": (C.c_int, [u64, vp, vp, C.POINTER(i32), vp, i64, i64, f64, C.POINTER(Rng), vp, vp, sz, vp]),
    "bk_smc_move_weight": (C.c_int, [u64, vp, i64, i32, i32, f64, C.POINTER(Rng), vp, vp, vp]),
    "bk_smc_gather_move_weight": (C.c_int, [u64, vp, vp, vp, i64, i32, i32, f64, C.POINTER(Rng), vp, vp, vp]),
    "bk_smc_gather_move_weight_acc": (C.c_int, [u64, vp, vp, vp, i64, i32, i32, f64, C.POINTER(Rng), vp, vp, vp, vp]),
    "bk_smc_adaptive_select": (C.c_int, [vp, f64, i64, i64, vp, vp, i32, vp, vp]),
    "bk_smc_resample_workspace_bytes": (sz, [i64]),
    "bk_smc_weight_stats": (C.c_int, [vp, i64, i32, i32, vp, vp, sz, vp]),
    "bk_smc_resample_indices": (C.c_int, [vp, i64, i32, i32, f64, f64, vp, C.POINTER(Rng), i64, i64,
                                          vp, vp, vp, sz, vp]),
    "bk_smc_resample_indices_dev": (C.c_int, [vp, i64, i32, i32, vp, vp, C.POINTER(Rng), i64, i64, vp, vp,
                                              vp, sz, vp]),
    "bk_gather_rows": (C.c_int, [vp, vp, i64, i64, i32, vp, vp]),
    "bk_smc_shard_workspace_bytes": (sz, [i64, i32, i32]),
    "bk_smc_shard_move": (C.c_int, [u64, C.POINTER(SmcShard), vp, i32, i32, C.POINTER(SmcKernel), C.POINTER(Rng), i32,
                                    vp, vp, sz, vp]),
    "bk_smc_shard_resample": (C.c_int, [C.POINTER(SmcShard), i32, i32, vp, C.POINTER(Rng), f64, i32, vp, vp, sz, vp]),
    "bk_smc_shard_run": (C.c_int, [u64, C.POINTER(SmcShard), vp, i32, i32, i32, C.POINTER(SmcKernel), C.POINTER(Rng), i32, f64,
                                   vp, vp, vp, sz, vp]),
    "bk_smc_cuda_prepare": (C.c_int, [u64, u64, C.c_char_p, sz]),
    "bk_smc_shard_gather": (C.c_int, [C.POINTER(SmcShard), i64, i32, vp, vp]),
    "bk_rank_normalize_workspace_bytes": (sz, [i64, i32]),
    "bk_rank_normalize": (C.c_int, [vp, i32, C.POINTER(SeriesLayout), vp, vp, vp, sz, vp]),
    "bk_autocorr_workspace_bytes": (sz, [i64, i64]),
    "bk_autocorr": (C.c_int, [vp, i32, C.POINTER(SeriesLayout), vp, vp, sz, vp]),
    "bk_iat_ess_workspace_bytes": (sz, [i32, C.POINTER(SeriesLayout)]),
    "bk_iat_ess": (C.c_int, [vp, i32, C.POINTER(SeriesLayout), i32, vp, vp, vp, sz, vp]),
    "bk_chain_moments": (C.c_int, [vp, i32, C.POINTER(SeriesLayout), vp, vp, vp]),
    "bk_moments_accumulate": (C.c_int, [vp, i32, i64, i64, i64, vp, vp, vp]),
    "bk_rhat_from_moments": (C.c_int, [vp, vp, vp, i64, i64, i64, vp, vp]),
    "bk_rhat_partial_sums": (C.c_int, [vp, vp, i64, i64, vp, vp, vp]),
    "bk_rhat_from_sums": (C.c_int, [vp, vp, i64, i64, vp, vp, vp]),
}

EXPORTS = tuple(_SIGNATURES)

_lib = None


def lib():
    """The loaded library (loads on first use; raises if it is not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BkError(
                f"{LIB_PATH} not found: the CUDA extension is not built. Run "
                "`python bayes-kit_b200/build.py` (or __graft_entry__.build()). There is no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        if l.bk_abi_version() != 1:
            raise BkError("libbk_b200.so ABI version mismatch")
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc == BK_OK:
        return
    msg = lib().bk_last_error().decode()
    if rc == BK_E_INVALID:
        raise ValueError(msg)
    if rc == BK_E_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise BkError(f"libbk_b200 error {rc}: {msg}")
