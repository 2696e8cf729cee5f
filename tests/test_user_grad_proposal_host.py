"""bk_proposal_create_cuda_grad without a GPU: the entry point is exported and declared, bad arguments are refused
before compiling, and two gradient proposals (MALA restated, and the Barker proposal) compile under NVRTC, on their
own and fused with a model.  The fused programs are compiled by _user_cuda.compile_program, a restatement of the
library's program text (user_model.cu: program_text and compile), checked first against the library's own compilation
of a proposal's and of a model's program; it also shows that a non-gradient proposal's programs hold the kernels they
always held."""
import ctypes as C

import pytest

from _user_cuda import (BANANA, BARKER, HEADER, MALA_G, PRIOR_LIK, PROGRAM_MODEL, PROGRAM_MODEL_PROPOSAL,
                        PROGRAM_PROPOSAL, RW, compile_program, entries, needs_nvrtc)
from bayes_kit_b200 import _lib

DUMMY_PTR = 256                                   # never dereferenced: validation and compilation do not touch params


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
@pytest.mark.parametrize("kind,gradient,f64,prior_lik", [
    (PROGRAM_PROPOSAL, False, False, False), (PROGRAM_PROPOSAL, True, False, False),
    (PROGRAM_MODEL, False, False, False), (PROGRAM_MODEL, False, True, False), (PROGRAM_MODEL, False, False, True),
], ids=["False", "True", "model", "model_f64", "model_prior_lik"])
def test_the_restated_program_text_is_the_librarys(kind, gradient, f64, prior_lik):
    """compile_program compiles what the library compiles: the same ptxas report for a proposal's own program (plain
    and gradient) and for a model's own program (plain, fp64, and a prior / likelihood pair with the SMC kernels).  The
    library compiles a model's program before loading it, so without a device it returns BK_E_CUDA with the log."""
    dtype = _lib.BK_F64 if f64 else _lib.BK_F32
    if kind == PROGRAM_PROPOSAL:
        src = MALA_G if gradient else RW
        rc, log, err = _create(src, 5, dtype, gradient=gradient)
        ok, mine = compile_program(kind, 5, f64, proposal=src, normals=5, transition=1, gradient=gradient)
    else:
        src = PRIOR_LIK if prior_lik else BANANA
        create = _lib.lib().bk_model_create_cuda_prior_lik if prior_lik else _lib.lib().bk_model_create_cuda
        h, buf = _lib.u64(0), C.create_string_buffer(1 << 20)
        rc = create(src.encode(), 5, dtype, DUMMY_PTR, 1, C.byref(h), buf, len(buf))
        if rc == _lib.BK_OK:
            _lib.lib().bk_model_destroy(h.value)
        log, err = buf.value.decode(), _lib.lib().bk_last_error().decode()
        ok, mine = compile_program(kind, 5, f64, model=src, prior_lik=prior_lik)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
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
    assert entries(log) == ["bk_user_dh_grad", "bk_user_propose_grad"]
    # without a transition there is no Hastings kernel
    rc, log, err = _create(src.split("__device__ bk_real transition_log_density")[0], D, dtype, uniforms=uniforms,
                           transition=0)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert entries(log) == ["bk_user_propose_grad"]
    # fused with the banana model, and with a prior / likelihood model (no SMC kernel for a gradient proposal)
    for model, pl in ((BANANA, False), (PRIOR_LIK, True)):
        ok, log = compile_program(PROGRAM_MODEL_PROPOSAL, D, f64, model, src, pl, normals=D, uniforms=uniforms,
                                  transition=1, gradient=True)
        assert ok, log
        assert entries(log) == ["bk_user_mhp_grad"]


@needs_nvrtc
@pytest.mark.parametrize("f64", [False, True])
def test_non_gradient_programs_hold_what_they_held(f64):
    dtype = _lib.BK_F64 if f64 else _lib.BK_F32
    rc, log, err = _create(RW, 8, dtype, gradient=False)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert entries(log) == ["bk_user_propose"]
    ok, log = compile_program(PROGRAM_MODEL_PROPOSAL, 8, f64, BANANA, RW, normals=8, transition=1)
    assert ok, log
    assert entries(log) == ["bk_user_mhp"]
    ok, log = compile_program(PROGRAM_MODEL_PROPOSAL, 8, f64, PRIOR_LIK, RW, True, normals=8, transition=1)
    assert ok, log
    assert entries(log) == ["bk_user_mhp", "bk_user_smc_mhp"]


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
