"""bk_drghmc_cuda_prepare without a GPU: the entry point is exported and declared, rejects an unknown handle, and a
model's own program does not contain DrGhmcDiag's kernel (that has a program of its own, compiled on first use)."""
import ctypes as C
import os

import pytest

from bayes_kit_b200 import _lib
from bayes_kit_b200.models import _load_nvrtc

HEADER = os.path.join(os.path.dirname(__file__), os.pardir, "include", "bk.h")

PLAIN = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; }
    return bk_real(-0.5) * s;
}
"""

PRIOR_LIK = """
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; }
    return bk_real(-0.5) * s;
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = x[e] - 1; s += d * d; g[e] = -d; }
    return bk_real(-0.5) * s;
}
"""


def _nvrtc_available():
    _load_nvrtc()
    try:
        C.CDLL("libnvrtc.so.12")
        return True
    except OSError:
        return False


def test_prepare_is_exported_and_declared():
    with open(HEADER) as f:
        assert "BK_API int bk_drghmc_cuda_prepare(uint64_t handle, char* log_out, size_t log_bytes);" in f.read()
    assert hasattr(_lib.lib(), "bk_drghmc_cuda_prepare")
    assert "bk_drghmc_cuda_prepare" in _lib.EXPORTS


def test_prepare_rejects_an_unknown_handle():
    log = C.create_string_buffer(b"stale", 64)
    rc = _lib.lib().bk_drghmc_cuda_prepare(987654321, log, len(log))
    assert rc == _lib.BK_E_HANDLE
    assert "987654321" in _lib.lib().bk_last_error().decode()
    assert log.value == b""


@pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC (libnvrtc.so.12) cannot be loaded")
@pytest.mark.parametrize("create,source", [("bk_model_create_cuda", PLAIN),
                                           ("bk_model_create_cuda_prior_lik", PRIOR_LIK)])
@pytest.mark.parametrize("dims", [2, 32])
def test_model_program_has_no_drghmc_kernel(create, source, dims):
    """BK_OK with a device, BK_E_CUDA (loading the module) without one; either way the log is the model program's."""
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 20)
    rc = getattr(_lib.lib(), create)(source.encode(), dims, _lib.BK_F32, None, 0, C.byref(h), log, len(log))
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), _lib.lib().bk_last_error().decode()
    if rc == _lib.BK_OK:
        _lib.lib().bk_model_destroy(h.value)
    text = log.value.decode()
    assert "bk_user_hmc" in text
    assert "bk_user_drghmc" not in text
