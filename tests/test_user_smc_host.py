"""bk_model_create_cuda_prior_lik without a GPU: argument validation and NVRTC compilation run before any device call,
so a broken source, or a broken embedded header (the SMC protocol header smc_mailbox.cuh, user_kernels.cuh's SMC
kernels), shows up here."""
import ctypes as C
import os

import pytest

from bayes_kit_b200 import _lib
from bayes_kit_b200.models import _load_nvrtc

# GaussPriorLik restated, params = [mu (D), pl (D), m0 (D), p0 (D)]
GPL = """
__device__ bk_real quad(const bk_real* x, bk_real* g, const bk_real* m, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = x[e] - m[e], pd = p[e] * d;
        s += pd * d;
        g[e] = -pd;
    }
    return bk_real(-0.5) * s;
}
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    return quad(x, g, p + 2 * BK_DIMS, p + 3 * BK_DIMS);
}
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    return quad(x, g, p, p + BK_DIMS);
}
"""

PLAIN = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; }
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


pytestmark = pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC (libnvrtc.so.12) cannot be loaded")

DUMMY_PTR = 256   # never dereferenced: validation and compilation do not touch params


def _create(source, dims, dtype=_lib.BK_F32, params=None, n_params=0, handle=True, fn="bk_model_create_cuda_prior_lik"):
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 18)
    src = None if source is None else source.encode()
    rc = getattr(_lib.lib(), fn)(src, dims, dtype, params, n_params, C.byref(h) if handle else None, log, len(log))
    if rc == _lib.BK_OK:
        _lib.lib().bk_model_destroy(h.value)
    return rc, log.value.decode(), _lib.lib().bk_last_error().decode()


@pytest.mark.parametrize("kw,msg", [
    (dict(source=None, dims=2), "source"),
    (dict(source=GPL, dims=2, handle=False), "handle_out"),
    (dict(source=GPL, dims=0), "dims"),
    (dict(source=GPL, dims=257), "dims"),
    (dict(source=GPL, dims=2, dtype=7), "dtype"),
    (dict(source=GPL, dims=2, params=None, n_params=8), "n_params"),
    (dict(source=GPL, dims=2, params=DUMMY_PTR, n_params=0), "n_params"),
    (dict(source=GPL, dims=2, params=DUMMY_PTR, n_params=-1), "n_params"),
])
def test_arguments_rejected_before_compiling(kw, msg):
    rc, log, err = _create(**kw)
    assert rc == _lib.BK_E_INVALID
    assert msg in err and "bk_model_create_cuda_prior_lik" in err
    assert log == ""


def test_dims_limit_is_the_header_constant():
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "bk.h")).read()
    assert "#define BK_USER_PRIOR_LIK_MAX_DIMS 256" in src
    rc, _, err = _create(GPL, 257)
    assert rc == _lib.BK_E_INVALID and "[1, 256]" in err


@pytest.mark.parametrize("dtype", [_lib.BK_F32, _lib.BK_F64])
@pytest.mark.parametrize("dims", [1, 5, 50])
def test_valid_source_gets_past_compilation(dims, dtype):
    """BK_OK with a device, BK_E_CUDA (loading the module) without one -- never BK_E_INVALID.  The log (ptxas's
    resource report) lists the prior/likelihood evaluator and the three SMC move kernels, which proves the shared
    mailbox header compiles under NVRTC; the fused MCMC kernels appear exactly when dims <= 32."""
    rc, log, err = _create(GPL, dims, dtype, DUMMY_PTR, 4 * dims)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    for k in ("bk_user_eval_pl", "bk_user_smc_rw", "bk_user_smc_mala", "bk_user_smc_hmc"):
        assert f"Function properties for {k}\n" in log, k
    assert ("bk_user_hmc" in log) == (dims <= 32)


def test_missing_likelihood_is_a_compile_error():
    src = GPL[:GPL.index("__device__ bk_real log_likelihood_gradient")]
    rc, log, err = _create(src, 3)
    assert rc == _lib.BK_E_INVALID
    assert "identifier \"log_likelihood_gradient\" is undefined" in log
    assert "compilation failed" in err and "\n" not in err


def test_plain_model_does_not_compile_the_smc_kernels():
    rc, log, err = _create(PLAIN, 5, fn="bk_model_create_cuda")
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert "bk_user_eval" in log
    assert "bk_user_smc" not in log and "bk_user_eval_pl" not in log


def test_prior_lik_source_is_not_a_plain_model():
    """The pair alone defines no log_density_gradient: only the prior/likelihood entry point derives it."""
    rc, log, _ = _create(GPL, 3, fn="bk_model_create_cuda")
    assert rc == _lib.BK_E_INVALID
    assert "identifier \"log_density_gradient\" is undefined" in log
