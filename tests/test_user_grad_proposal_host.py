"""bk_proposal_create_cuda_grad without a GPU: the entry point is exported and declared, bad arguments are refused
before compiling, and two gradient proposals (MALA restated, and the Barker proposal) compile under NVRTC, on their
own and fused with a model.  The fused programs are compiled here by a restatement of the library's program text
(user_model.cu: program_text and compile), checked first against the library's own compilation of a proposal
program; it also shows that a non-gradient proposal's programs hold the kernels they always held."""
import ctypes as C
import os
import re

import pytest

from bayes_kit_b200 import _lib
from bayes_kit_b200.models import _load_nvrtc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bayes-kit_b200", "csrc")
HEADER = os.path.join(ROOT, "include", "bk.h")

# MALA as a gradient proposal, params = [eps, sqrt(2 eps), -1 / (4 eps)]
MALA_G = """
__device__ void propose(const bk_real* th, const bk_real* g, bk_real* q, const bk_real* z, const bk_real* u,
                        const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = th[e] + p[0] * g[e] + p[1] * z[e];
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* gf,
                                          const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = to[e] - from[e] - p[0] * gf[e]; s += d * d; }
    return p[2] * s;
}
"""

# the Barker proposal (Livingstone & Zanella 2022), params = [sigma]: w_e = sigma z_e, kept with probability
# 1 / (1 + exp(-w_e g_e)) and flipped otherwise (u_e, one uniform per coordinate)
BARKER = """
__device__ bk_real softplus(bk_real x) { return x > 0 ? x + log1p(exp(-x)) : log1p(exp(x)); }
__device__ void propose(const bk_real* th, const bk_real* g, bk_real* q, const bk_real* z, const bk_real* u,
                        const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real w = p[0] * z[e];
        const bk_real keep = 1 / (1 + exp(-w * g[e]));
        q[e] = th[e] + (u[e] < keep ? w : -w);
    }
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* gf,
                                          const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        const bk_real w = to[e] - from[e], r = w / p[0];
        s -= bk_real(0.5) * r * r + softplus(-w * gf[e]);
    }
    return s;
}
"""

# a plain random walk (non-gradient signatures)
RW = """
__device__ void propose(const bk_real* theta, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {
    for (int e = 0; e < BK_DIMS; ++e) q[e] = theta[e] + p[0] * z[e];
}
__device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* p) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) { const bk_real d = to[e] - from[e]; s += d * d; }
    return bk_real(-0.5) * s / (p[0] * p[0]);
}
"""

BANANA = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
    const bk_real b = params[0], half = 0.5, two = 2;
    const bk_real u = x[1] - b * x[0] * x[0];
    bk_real lp = -half * (x[0] * x[0]) - half * (u * u);
    g[0] = -x[0] + two * b * x[0] * u;
    g[1] = -u;
    for (int e = 2; e < BK_DIMS; ++e) {
        lp -= half * (x[e] * x[e]);
        g[e] = -x[e];
    }
    return lp;
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

PROGRAM_PROPOSAL, PROGRAM_MODEL_PROPOSAL = 2, 3   # BK_PROGRAM_* (user_kernels.cuh)
DUMMY_PTR = 256                                   # never dereferenced: validation and compilation do not touch params


def _nvrtc():
    _load_nvrtc()
    try:
        return C.CDLL("libnvrtc.so.12")
    except OSError:
        return None


needs_nvrtc = pytest.mark.skipif(_nvrtc() is None, reason="NVRTC (libnvrtc.so.12) cannot be loaded")


def _entries(log):
    """the kernels ptxas reports, sorted"""
    return sorted(re.findall(r"Compiling entry function '(\w+)'", log))


def _create(source, dims, dtype=_lib.BK_F32, params=DUMMY_PTR, n_params=1, normals=None, uniforms=0, transition=1,
            gradient=True, handle=True):
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 20)
    src = None if source is None else source.encode()
    fn = _lib.lib().bk_proposal_create_cuda_grad if gradient else _lib.lib().bk_proposal_create_cuda
    rc = fn(src, dims, dtype, params, n_params, dims if normals is None else normals, uniforms, transition,
            C.byref(h) if handle else None, log, len(log))
    if rc == _lib.BK_OK:
        assert h.value >> 62 == 1
        assert _lib.lib().bk_proposal_destroy(h.value) == _lib.BK_OK
    return rc, log.value.decode(), _lib.lib().bk_last_error().decode()


def _program(kind, D, f64, proposal, normals, uniforms, transition, gradient, model=None, prior_lik=False):
    """NVRTC compile of the text user_model.cu builds for a program of `kind`; returns (ok, log)."""
    read = lambda name: open(os.path.join(CSRC, name)).read()   # noqa: E731
    smc = prior_lik and not gradient and kind == PROGRAM_MODEL_PROPOSAL
    text = ("typedef unsigned int uint32_t;\ntypedef unsigned long long uint64_t;\n"
            "typedef int int32_t;\ntypedef long long int64_t;\n")
    text += '#line 1 "bk_device_rng.cuh"\n' + read("device_rng.cuh")
    text += "\ntypedef double bk_real;\n" if f64 else "\ntypedef float bk_real;\n"
    if model:
        text += '#line 1 "model.cu"\n' + model
        if smc:
            text += '\n#line 1 "bk_smc_mailbox.cuh"\n' + read("smc_mailbox.cuh")
    text += '\nnamespace bk_proposal {\n#line 1 "proposal.cu"\n' + proposal + "\n}  // namespace bk_proposal\n"
    text += '\n#line 1 "bk_user_kernels.cuh"\n' + read("user_kernels.cuh")
    opts = ["-arch=sm_100a", "-std=c++17", f"-DBK_PROGRAM={kind}", f"-DBK_DIMS={D}", "-DBK_USER_FUSED_MAX_D=32",
            "--ptxas-options=-v"]
    if f64:
        opts.append("--fmad=false")
    if prior_lik:
        opts.append("-DBK_PRIOR_LIK=1")
    if smc:
        opts += ["-DBK_SMC_KERNELS=1", "-DBK_SMC_MAX_WORLD=16", "-DBK_SMC_MAILBOX_BYTES=4096"]
    opts += [f"-DBK_PROPOSAL_NORMALS={normals}", f"-DBK_PROPOSAL_UNIFORMS={uniforms}",
             f"-DBK_PROPOSAL_TRANSITION={transition}"]
    if gradient:
        opts.append("-DBK_PROPOSAL_GRADIENT=1")
    nv = _nvrtc()
    prog = C.c_void_p()
    name = b"proposal.cu" if kind == PROGRAM_PROPOSAL else b"model.cu"
    assert nv.nvrtcCreateProgram(C.byref(prog), text.encode(), name, 0, None, None) == 0
    arr = (C.c_char_p * len(opts))(*[o.encode() for o in opts])
    rc = nv.nvrtcCompileProgram(prog, len(opts), arr)
    n = C.c_size_t(0)
    nv.nvrtcGetProgramLogSize(prog, C.byref(n))
    buf = C.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(prog, buf)
    nv.nvrtcDestroyProgram(C.byref(prog))
    return rc == 0, buf.value.decode()


def test_entry_point_is_exported_and_declared():
    with open(HEADER) as f:
        assert "BK_API int bk_proposal_create_cuda_grad(" in f.read()
    assert hasattr(_lib.lib(), "bk_proposal_create_cuda_grad")
    assert "bk_proposal_create_cuda_grad" in _lib.EXPORTS


@needs_nvrtc
@pytest.mark.parametrize("kw,msg", [
    (dict(source=None, dims=2), "source"),
    (dict(source=MALA_G, dims=2, handle=False), "handle_out"),
    (dict(source=MALA_G, dims=0), "dims"),
    (dict(source=MALA_G, dims=65537, normals=1), "dims"),
    (dict(source=MALA_G, dims=2, dtype=7), "dtype"),
    (dict(source=MALA_G, dims=2, params=None, n_params=1), "n_params"),
    (dict(source=MALA_G, dims=2, params=DUMMY_PTR, n_params=0), "n_params"),
    (dict(source=MALA_G, dims=2, normals=-1), "n_normals"),
    (dict(source=MALA_G, dims=2, uniforms=65), "n_uniforms"),
])
def test_arguments_rejected_before_compiling(kw, msg):
    rc, log, err = _create(**kw)
    assert rc == _lib.BK_E_INVALID
    assert msg in err and "bk_proposal_create_cuda_grad" in err
    assert log == ""


@needs_nvrtc
@pytest.mark.parametrize("gradient", [False, True])
def test_the_restated_program_text_is_the_librarys(gradient):
    """The harness below compiles what the library compiles: the same ptxas report for a proposal's own program."""
    src = MALA_G if gradient else RW
    rc, log, err = _create(src, 5, gradient=gradient)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    ok, mine = _program(PROGRAM_PROPOSAL, 5, False, src, 5, 0, 1, gradient)
    assert ok, mine
    lines = lambda s: [ln for ln in s.splitlines() if ln.startswith("ptxas") and "time" not in ln]   # noqa: E731
    assert lines(mine) == lines(log) and lines(log)


@needs_nvrtc
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("D", [2, 16, 32])
@pytest.mark.parametrize("name", ["mala", "barker"])
def test_gradient_proposals_compile(name, D, f64):
    src, uniforms = (MALA_G, 0) if name == "mala" else (BARKER, D)
    dtype = _lib.BK_F64 if f64 else _lib.BK_F32
    # the proposal's own program (the three-launch path), through the library
    rc, log, err = _create(src, D, dtype, uniforms=uniforms)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert _entries(log) == ["bk_user_dh_grad", "bk_user_propose_grad"]
    # without a transition there is no Hastings kernel
    rc, log, err = _create(src.split("__device__ bk_real transition_log_density")[0], D, dtype, uniforms=uniforms,
                           transition=0)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert _entries(log) == ["bk_user_propose_grad"]
    # fused with the banana model, and with a prior / likelihood model (no SMC kernel for a gradient proposal)
    for model, pl in ((BANANA, False), (PRIOR_LIK, True)):
        ok, log = _program(PROGRAM_MODEL_PROPOSAL, D, f64, src, D, uniforms, 1, True, model, pl)
        assert ok, log
        assert _entries(log) == ["bk_user_mhp_grad"]


@needs_nvrtc
@pytest.mark.parametrize("f64", [False, True])
def test_non_gradient_programs_hold_what_they_held(f64):
    dtype = _lib.BK_F64 if f64 else _lib.BK_F32
    rc, log, err = _create(RW, 8, dtype, gradient=False)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert _entries(log) == ["bk_user_propose"]
    ok, log = _program(PROGRAM_MODEL_PROPOSAL, 8, f64, RW, 8, 0, 1, False, BANANA)
    assert ok, log
    assert _entries(log) == ["bk_user_mhp"]
    ok, log = _program(PROGRAM_MODEL_PROPOSAL, 8, f64, RW, 8, 0, 1, False, PRIOR_LIK, True)
    assert ok, log
    assert _entries(log) == ["bk_user_mhp", "bk_user_smc_mhp"]


@needs_nvrtc
@pytest.mark.parametrize("source,diag", [
    # a proposal with the non-gradient signature is not a gradient proposal
    (RW, "propose"),
    ("\n__device__ void propose(const bk_real* t, const bk_real* g, bk_real* q, const bk_real* z, const bk_real* u,"
     " const bk_real* p) { q[0] = t[0] }", "proposal.cu(2): error"),
])
def test_compile_error_returns_the_log(source, diag):
    rc, log, err = _create(source, 3, transition=0)
    assert rc == _lib.BK_E_INVALID
    assert diag in log and "error" in log
    assert "bk_proposal_create_cuda_grad: compilation failed" in err
