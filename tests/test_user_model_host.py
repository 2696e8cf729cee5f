"""bk_model_create_cuda without a GPU: argument validation and NVRTC compilation run before any device call, so a
broken source, a broken embedded header (device_rng.cuh) or a broken kernel file (user_kernels.cuh) shows up here."""
import ctypes as C

import pytest

from bayes_kit_b200 import _lib
from bayes_kit_b200.models import _load_nvrtc

BANANA = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
    const bk_real b = params[0], half = 0.5, two = 2;
    const bk_real u = x[1] - b * x[0] * x[0];
    bk_real lp = -half * (x[0] * x[0]) - half * (u * u);
    g[0] = -x[0] + two * b * x[0] * u;
    g[1] = -u;
    for (int e = 2; e < BK_DIMS; ++e) { lp -= half * (x[e] * x[e]); g[e] = -x[e]; }
    return lp;
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


def _create(source, dims, dtype=_lib.BK_F32, params=None, n_params=0, handle=True):
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 16)
    src = None if source is None else source.encode()
    rc = _lib.lib().bk_model_create_cuda(src, dims, dtype, params, n_params, C.byref(h) if handle else None,
                                         log, len(log))
    if rc == _lib.BK_OK:
        _lib.lib().bk_model_destroy(h.value)
    return rc, log.value.decode(), _lib.lib().bk_last_error().decode()


@pytest.mark.parametrize("kw,msg", [
    (dict(source=None, dims=2), "source"),
    (dict(source=BANANA, dims=2, handle=False), "handle_out"),
    (dict(source=BANANA, dims=0), "dims"),
    (dict(source=BANANA, dims=65537), "dims"),
    (dict(source=BANANA, dims=2, dtype=7), "dtype"),
    (dict(source=BANANA, dims=2, params=None, n_params=1), "n_params"),
    (dict(source=BANANA, dims=2, params=DUMMY_PTR, n_params=0), "n_params"),
    (dict(source=BANANA, dims=2, params=DUMMY_PTR, n_params=-1), "n_params"),
])
def test_arguments_rejected_before_compiling(kw, msg):
    rc, log, err = _create(**kw)
    assert rc == _lib.BK_E_INVALID
    assert msg in err
    assert log == ""


@pytest.mark.parametrize("source,diag", [
    # diagnostics in the user's source carry its own line numbers
    ("__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) { return x[0] }",
     "model.cu(1): error: expected a \";\""),
    ("__device__ bk_real log_density(const bk_real* x, const bk_real* p) { return -x[0] * x[0]; }",
     "error: identifier \"log_density_gradient\" is undefined"),
])
def test_compile_error_returns_the_log(source, diag):
    rc, log, err = _create(source, 3)
    assert rc == _lib.BK_E_INVALID
    assert diag in log
    assert "compilation failed" in err and "\n" not in err


@pytest.mark.parametrize("dtype", [_lib.BK_F32, _lib.BK_F64])
@pytest.mark.parametrize("dims", [2, 17, 100])
def test_valid_source_gets_past_compilation(dims, dtype):
    """BK_OK with a device, BK_E_CUDA (loading the module) without one -- never BK_E_INVALID.  dims 2 and 17 compile
    the fused samplers too, 100 only the evaluation kernel."""
    rc, log, err = _create(BANANA, dims, dtype, DUMMY_PTR, 1)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert "bk_user_eval" in log                       # ptxas's resource report of every kernel
    assert ("bk_user_hmc" in log) == (dims <= 32)
