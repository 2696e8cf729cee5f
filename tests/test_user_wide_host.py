"""The wide HMCDiag / MALA / RW-Metropolis program of user models (BK_PROGRAM_WIDE) without a GPU.

Without a device no model handle exists (loading a model's module needs one), so the program is compiled here the way
user_model.cu compiles it: the same text (the library's device header, the model's source, user_kernels.cuh) and the
same NVRTC options.  ptxas's report must list the three kernels, with no spill stores for the banana and the diagonal
Gaussian in fp32 at every D in range.  The prepare entry point itself is checked for its declaration and for an
unknown handle; with handles (on the GPU) tests/test_gpu_user_wide.py checks the rest."""
import ctypes as C
import os
import re

import pytest

from bayes_kit_b200 import _lib
from bayes_kit_b200.models import _load_nvrtc

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), os.pardir)
CSRC = os.path.join(ROOT, "bayes-kit_b200", "csrc")
HEADER = os.path.join(ROOT, "include", "bk.h")


def _define(name):
    with open(os.path.join(CSRC, "model.h")) as f:
        return int(re.search(rf"#define {name} (\d+)", f.read()).group(1))


FUSED_MAX_D = _define("BK_USER_FUSED_MAX_D")
WIDE_MAX_D = _define("BK_USER_WIDE_MAX_D")
PROGRAM_WIDE = 6
KERNELS = ("bk_user_wide_hmc", "bk_user_wide_mala", "bk_user_wide_mh")

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

DIAG = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real d = x[e] - p[e];
        const bk_real pd = p[BK_DIMS + e] * d;
        s += d * pd;
        g[e] = -pd;
    }
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
SOURCES = {"banana": BANANA, "diag": DIAG, "prior_lik": PRIOR_LIK}


def _nvrtc():
    _load_nvrtc()
    try:
        return C.CDLL("libnvrtc.so.12")
    except OSError:
        return None


pytestmark = pytest.mark.skipif(_nvrtc() is None, reason="NVRTC (libnvrtc.so.12) cannot be loaded")


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def compile_wide(source, dims, f64, prior_lik):
    """(NVRTC result, log) of the wide program: program_text() and compile() of user_model.cu."""
    nv = _nvrtc()
    text = ("typedef unsigned int uint32_t;\ntypedef unsigned long long uint64_t;\n"
            "typedef int int32_t;\ntypedef long long int64_t;\n"
            "#line 1 \"bk_device_rng.cuh\"\n" + _read("device_rng.cuh") +
            ("\ntypedef double bk_real;\n" if f64 else "\ntypedef float bk_real;\n") +
            "#line 1 \"model.cu\"\n" + source +
            "\n#line 1 \"bk_user_kernels.cuh\"\n" + _read("user_kernels.cuh"))
    opts = ["-arch=sm_100a", "-std=c++17", f"-DBK_PROGRAM={PROGRAM_WIDE}", f"-DBK_DIMS={dims}",
            f"-DBK_USER_FUSED_MAX_D={FUSED_MAX_D}", "--ptxas-options=-v"]
    if f64:
        opts.append("--fmad=false")
    if prior_lik:
        opts.append("-DBK_PRIOR_LIK=1")
    opts.append("-DBK_WIDE=1")
    prog = C.c_void_p()
    assert nv.nvrtcCreateProgram(C.byref(prog), text.encode(), b"model.cu", 0, None, None) == 0
    arr = (C.c_char_p * len(opts))(*[o.encode() for o in opts])
    rc = nv.nvrtcCompileProgram(prog, len(opts), arr)
    n = C.c_size_t()
    nv.nvrtcGetProgramLogSize(prog, C.byref(n))
    buf = C.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(prog, buf)
    nv.nvrtcDestroyProgram(C.byref(prog))
    return rc, buf.value.decode()


def ptxas_report(log):
    """kernel -> (registers, spill store bytes, spill load bytes, shared bytes)"""
    out = {}
    for k in KERNELS:
        m = re.search(rf"Function properties for {k}\n.*?(\d+) bytes spill stores, (\d+) bytes spill loads\n"
                      rf".*?Used (\d+) registers", log, re.S)
        if m:
            out[k] = (int(m.group(3)), int(m.group(1)), int(m.group(2)))
    return out


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
    rc, log = compile_wide(SOURCES[which], dims, f64, which == "prior_lik")
    assert rc == 0, log
    rep = ptxas_report(log)
    assert set(rep) == set(KERNELS), log
    if which != "prior_lik" and not f64:
        for k, (_, spill_st, _) in rep.items():
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
