"""The wide HMCDiag / MALA / RW-Metropolis program of user models (BK_PROGRAM_WIDE) without a GPU.

Without a device no model handle exists (loading a model's module needs one), so the program is compiled by
_user_cuda.compile_program the way user_model.cu compiles it: the same text (the library's device header, the model's
source, user_kernels.cuh) and the same NVRTC options.  ptxas's report must list the three kernels, with no spill
stores for the banana and the diagonal Gaussian in fp32 at every D in range.  The prepare entry point itself is
checked for its declaration and for an unknown handle; with handles (on the GPU) tests/test_gpu_user_wide.py checks
the rest."""
import ctypes as C

import pytest

from _user_cuda import (BANANA, DIAG, FUSED_MAX_D, HEADER, PRIOR_LIK, PROGRAM_WIDE, WIDE_MAX_D, compile_program,
                        needs_nvrtc, ptxas_report)
from bayes_kit_b200 import _lib

KERNELS = ("bk_user_wide_hmc", "bk_user_wide_mala", "bk_user_wide_mh")
SOURCES = {"banana": BANANA, "diag": DIAG, "prior_lik": PRIOR_LIK}
pytestmark = needs_nvrtc


def test_prepare_is_exported_and_declared():
    with open(HEADER) as f:
        assert "BK_API int bk_user_wide_prepare(uint64_t model, char* log_out, size_t log_bytes);" in f.read()
    assert hasattr(_lib.lib(), "bk_user_wide_prepare")
    assert "bk_user_wide_prepare" in _lib.EXPORTS


def test_prepare_rejects_an_unknown_handle():
    log = C.create_string_buffer(b"stale", 64)
    rc = _lib.lib().bk_user_wide_prepare(987654321, log, len(log))
    assert rc == _lib.BK_E_HANDLE
    assert "987654321" in _lib.lib().bk_last_error().decode()
    assert log.value == b""


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("dims", sorted({33, 64, 128, WIDE_MAX_D}))
@pytest.mark.parametrize("which", ["banana", "diag", "prior_lik"])
def test_wide_program_compiles(which, dims, f64):
    ok, log = compile_program(PROGRAM_WIDE, dims, f64, SOURCES[which], prior_lik=which == "prior_lik")
    assert ok, log
    rep = ptxas_report(log)
    assert set(rep) == set(KERNELS), log
    if which != "prior_lik" and not f64:
        for k, r in rep.items():
            spill_st = r["spill_store_bytes"]
            assert spill_st == 0, (k, rep[k])


@pytest.mark.parametrize("dims", [FUSED_MAX_D + 1, WIDE_MAX_D])
def test_model_program_has_no_wide_kernel(dims):
    """The model's own program is that of every other model: the wide kernels are compiled in a program of their
    own.  BK_OK with a device, BK_E_CUDA (loading the module) without one; either way the log is the model's."""
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 20)
    rc = _lib.lib().bk_model_create_cuda(BANANA.encode(), dims, _lib.BK_F32, 256, 1, C.byref(h), log, len(log))
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), _lib.lib().bk_last_error().decode()
    if rc == _lib.BK_OK:
        _lib.lib().bk_model_destroy(h.value)
    text = log.value.decode()
    assert "bk_user_eval" in text
    assert "bk_user_wide" not in text
