"""bk_stretch_cuda_prepare without a GPU: the entry point is exported and declared, rejects an unknown handle, and a
model's own program does not contain the Stretcher's kernel (that has a program of its own, compiled on first use)."""
import ctypes as C

import pytest

from _user_cuda import HEADER, PLAIN, PRIOR_LIK, needs_nvrtc
from bayes_kit_b200 import _lib


def test_prepare_is_exported_and_declared():
    with open(HEADER) as f:
        assert "BK_API int bk_stretch_cuda_prepare(uint64_t handle, char* log_out, size_t log_bytes);" in f.read()
    assert hasattr(_lib.lib(), "bk_stretch_cuda_prepare")
    assert "bk_stretch_cuda_prepare" in _lib.EXPORTS


def test_prepare_rejects_an_unknown_handle():
    log = C.create_string_buffer(b"stale", 64)
    rc = _lib.lib().bk_stretch_cuda_prepare(987654321, log, len(log))
    assert rc == _lib.BK_E_HANDLE
    assert "987654321" in _lib.lib().bk_last_error().decode()
    assert log.value == b""


@needs_nvrtc
@pytest.mark.parametrize("create,source", [("bk_model_create_cuda", PLAIN),
                                           ("bk_model_create_cuda_prior_lik", PRIOR_LIK)])
def test_model_program_has_no_stretch_kernel(create, source):
    """BK_OK with a device, BK_E_CUDA (loading the module) without one; either way the log is the model program's."""
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 20)
    rc = getattr(_lib.lib(), create)(source.encode(), 8, _lib.BK_F32, None, 0, C.byref(h), log, len(log))
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), _lib.lib().bk_last_error().decode()
    if rc == _lib.BK_OK:
        _lib.lib().bk_model_destroy(h.value)
    text = log.value.decode()
    assert "bk_user_hmc" in text
    assert "bk_user_stretch" not in text
