"""Several MCMC moves per SMC temperature (TemperedLikelihoodSMC(..., moves=k)) without a GPU: the bk_smc_kernel layout
the ctypes binding assumes, the new entry point and its handle checks, the argument check of the Python constructor,
the composed-kernel restatement against the reference's recorded runs, the Philox block-offset rule, and NVRTC compiling
the SMC_MOVES program kind."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import _smc_moves_oracle as mo
import _user_cuda as uc
from bayes_kit_b200 import _lib
from conftest import golden
from oracle import philox as ph
from oracle import samplers as osm
from oracle.models import GaussPriorLik, build_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROGRAM_SMC_MOVES = 7

_LAYOUT = r"""
#include <stddef.h>
#include <stdio.h>
#include "bk.h"
int main() {
    printf("%zu %zu %zu %zu %zu %zu %d\n", sizeof(bk_smc_kernel), offsetof(bk_smc_kernel, kind),
           offsetof(bk_smc_kernel, steps), offsetof(bk_smc_kernel, scale), offsetof(bk_smc_kernel, proposal),
           offsetof(bk_smc_kernel, moves), (int)BK_SMC_MAX_MOVES);
    return 0;
}
"""


def _compiler():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand) and os.access(cand, os.X_OK):
            return cand
    return None


def test_smc_kernel_layout_with_moves_matches_bk_h(tmp_path):
    cc = _compiler()
    if cc is None:
        pytest.skip("no nvcc")
    src, exe = tmp_path / "layout.cu", tmp_path / "layout"
    src.write_text(_LAYOUT)
    r = subprocess.run([cc, f"-I{os.path.join(ROOT, 'include')}", str(src), "-o", str(exe)], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    K = _lib.SmcKernel
    assert got == [C.sizeof(K), K.kind.offset, K.steps.offset, K.scale.offset, K.proposal.offset, K.moves.offset,
                   _lib.SMC_MAX_MOVES]
    # initialisers of the existing kinds leave moves at 0, which means one move
    assert _lib.SmcKernel(_lib.SMC_KERNEL_RW, 0, 0.2).moves == 0


def test_prepare_is_exported_and_declared():
    assert "bk_smc_moves_prepare" in _lib.EXPORTS
    with open(os.path.join(ROOT, "include", "bk.h")) as f:
        h = f.read()
    assert re.search(r"BK_API int bk_smc_moves_prepare\(uint64_t model, const bk_smc_kernel\* kernel, char\* log_out, "
                     r"size_t log_bytes\);", h)
    assert re.search(r"#define BK_SMC_MAX_MOVES 65535\b", h)


def test_unknown_handles_are_refused_before_any_device_call():
    lib = _lib.lib()
    log = C.create_string_buffer(64)
    log.value = b"stale"
    kn = _lib.SmcKernel(_lib.SMC_KERNEL_RW, 0, 0.2, 0, 3)
    assert lib.bk_smc_moves_prepare(12345, C.byref(kn), log, len(log)) == _lib.BK_E_HANDLE
    assert log.value == b""
    assert lib.bk_smc_moves_prepare(0, None, None, 0) == _lib.BK_E_HANDLE
    kp = _lib.SmcKernel(_lib.SMC_KERNEL_PROPOSAL, 0, 0.0, 1 << 62, 3)
    assert lib.bk_smc_moves_prepare(12345, C.byref(kp), None, 0) == _lib.BK_E_HANDLE
    sh, rng = _lib.SmcShard(), _lib.Rng()
    assert lib.bk_smc_shard_move(12345, C.byref(sh), None, 1, 1, C.byref(kn), C.byref(rng), 0, None, None, 0,
                                 None) == _lib.BK_E_HANDLE


@pytest.mark.parametrize("moves", [0, -1, 65536, 2.5, True, "3"])
def test_moves_out_of_range_is_a_value_error(bk, moves):
    # checked before anything touches the model or the device
    with pytest.raises(ValueError, match="moves"):
        bk.TemperedLikelihoodSMC(None, 8, 2, np.zeros((8, 1)), bk.metropolis_kernel(0.2), moves=moves)


# ---- oracle ---------------------------------------------------------------------------------------------------------
def _extra_identity_moves(z, k, u_extra=0.5):
    """the golden streams as move 0 of k moves; moves 1..k-1 get zero normals (the walk stays put)"""
    T, M, D = z["normals"].shape
    zs = np.zeros((T, M, k, D))
    zs[:, :, 0] = z["normals"]
    au = np.full((T, M, k), u_extra)
    au[:, :, 0] = z["acc_uniforms"]
    return zs, au


@pytest.mark.parametrize("k", [2, 5])
@pytest.mark.parametrize("name", ["smc_gauss_d5", "smc_gauss_d50", "smc_binom"])
def test_zero_extra_normals_reproduce_the_rw_goldens(name, k):
    z = golden(name)
    model, s, T = build_model(z), float(z["scale"]), int(z["T"])
    zs, au = _extra_identity_moves(z, k)
    th, idx, _ = mo.smc_tempered(model, z["thetas0"], zs, au, z["res_uniforms"], T, ("rw", s))
    assert np.array_equal(idx, z["indices"])
    one, one_idx = osm.smc_tempered(model, z["thetas0"], z["normals"], z["acc_uniforms"], z["res_uniforms"], s, T)
    assert np.array_equal(th, one) and np.array_equal(idx, one_idx)
    np.testing.assert_allclose(th, z["thetas_final"], rtol=1e-10, atol=1e-10)
    # the proposal move with the walk restated: the same run
    walk = lambda t, zz, u: t + s * zz
    thp, idxp, accp = mo.smc_tempered_proposal(model, z["thetas0"], zs, au, z["res_uniforms"], T, walk)
    assert np.array_equal(thp, th) and np.array_equal(idxp, idx)
    assert accp.min() >= k - 1 and accp.max() <= k   # the identity moves always accept
    # one move per temperature through the multi-move restatement is the pinned single-move oracle
    th1, idx1, _ = mo.smc_tempered(model, z["thetas0"], z["normals"][:, :, None], z["acc_uniforms"][:, :, None],
                                   z["res_uniforms"], T, ("rw", s))
    assert np.array_equal(th1, one) and np.array_equal(idx1, one_idx)


@pytest.mark.parametrize("kernel", [("rw", 0.4), ("mala", 0.05), ("hmc", 0.1, 3)])
@pytest.mark.parametrize("resample", ["multinomial", "systematic"])
def test_moves_equal_an_explicit_loop_of_smc_move(kernel, resample):
    rng = np.random.default_rng(5)
    D, M, T, k = 3, 24, 4, 3
    mu = rng.normal(size=D)
    model = GaussPriorLik(np.zeros(D), np.ones(D), mu, 4 * np.ones(D))
    th0 = rng.normal(size=(M, D))
    zs, au, ru = rng.standard_normal((T, M, k, D)), rng.random((T, M, k)), rng.random((T, M))
    got, gidx, gacc = mo.smc_tempered(model, th0, zs, au, ru, T, kernel, resample=resample)
    assert gacc.min() >= 0 and gacc.max() <= k and gacc.sum() > 0
    th = th0.copy()
    for n in range(1, T + 1):
        t0, t1 = (n - 1) / T, n / T
        for m in range(M):
            for j in range(k):
                th[m] = osm.smc_move(model, th[m], t0, zs[n - 1, m, j], au[n - 1, m, j], kernel)
        if resample == "multinomial":
            idx, _ = osm.multinomial_indices(osm.smc_weights(model, th, n, T), ru[n - 1])
        else:
            lw = np.array([(model.log_likelihood(t) * t1 + model.log_prior(t)) -
                           (model.log_likelihood(t) * t0 + model.log_prior(t)) for t in th])
            idx, _ = osm.systematic_indices(lw, ru[n - 1, 0])
        assert np.array_equal(idx, gidx[n - 1])
        th = th[idx]
    assert np.array_equal(th, got)


def test_adaptive_restatement_with_moves_is_the_composed_walk():
    rng = np.random.default_rng(8)
    D, M, T, k, s = 4, 40, 6, 2, 0.3
    model = GaussPriorLik(np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D))
    th0 = rng.normal(size=(M, D))
    zs, au, ru = rng.standard_normal((T, M, k, D)), rng.random((T, M, k)), rng.random((T, M))
    th, lw, fl = mo.smc_tempered_adaptive(model, th0, zs, au, ru, T, 0.6, ("rw", s))
    # with zero normals in move 1 the two-move run is the pinned one-move oracle's run
    z1 = zs.copy()
    z1[:, :, 1] = 0.0
    a, la, fa = mo.smc_tempered_adaptive(model, th0, z1, au, ru, T, 0.6, ("rw", s))
    b, lb, fb = osm.smc_tempered_adaptive(model, th0, zs[:, :, 0], au[:, :, 0], ru, s, T, 0.6)
    assert np.array_equal(a, b) and np.array_equal(la, lb) and np.array_equal(fa, fb)
    assert not np.array_equal(th, a)


# ---- Philox block-offset rule -----------------------------------------------------------------------------------------
def test_move_streams_follow_the_block_offset_rule():
    seed, chain, draw = 0x1234ABCD5678, np.arange(7, dtype=np.uint64) + 100, 9
    assert mo.smc_move_block(0) == 0 and mo.smc_move_block(3) == 3 << 16
    D = 50
    ub = ph.accept_block(D)
    for j in range(4):
        b = mo.smc_move_block(j)
        # move j's words are move 0's words at block b + 2^16 j, for the normals, the accept uniform and TAG_UNIFORM
        np.testing.assert_array_equal(ph.normal4_f64(seed, 2 + b, chain, draw),
                                      ph.normal4_f64(seed, np.uint64(2 + (j << 16)), chain, draw))
        w = ph.gen(seed, ub + b, ph.TAG_NORMAL, chain, draw)
        want = ph.u01d(w[0], w[1])
        if j == 0:
            np.testing.assert_array_equal(want, ph.accept_uniform(seed, chain, draw, D, np.float64))
        else:
            assert not np.array_equal(want, ph.accept_uniform(seed, chain, draw, D, np.float64))
        for k in (0, 5, 63):
            u = ph.philox_uniform(seed, k + (j << 18), chain, draw, np.float32)    # fp32: block k >> 2
            v = ph.philox_uniform(seed, k + (j << 17), chain, draw, np.float64)    # fp64: block k >> 1
            wf = ph.gen(seed, (k >> 2) + b, ph.TAG_UNIFORM, chain, draw)
            wd = ph.gen(seed, (k >> 1) + b, ph.TAG_UNIFORM, chain, draw)
            np.testing.assert_array_equal(u, ph.u01(wf[k & 3]))
            np.testing.assert_array_equal(v, ph.u01d(wd[2], wd[3]) if k & 1 else ph.u01d(wd[0], wd[1]))
    # every block a single move uses lies below 2^16: 256 dims, 512 proposal normals, 64 uniforms
    assert ph.accept_block(256) < 1 << 16 and (512 // 4 + 1) < 1 << 16 and (64 >> 1) < 1 << 16


# ---- NVRTC: the SMC_MOVES program kind --------------------------------------------------------------------------------
def _compile_moves(D, f64, model, proposal=None, normals=0, uniforms=0, transition=0):
    """(ok, log) of NVRTC compiling a prior/likelihood model's SMC_MOVES program as user_model.cu does"""
    text = ("typedef unsigned int uint32_t;\ntypedef unsigned long long uint64_t;\n"
            "typedef int int32_t;\ntypedef long long int64_t;\n")
    text += '#line 1 "bk_device_rng.cuh"\n' + uc._read("device_rng.cuh")
    text += "\ntypedef double bk_real;\n" if f64 else "\ntypedef float bk_real;\n"
    text += '#line 1 "model.cu"\n' + model + '\n#line 1 "bk_smc_mailbox.cuh"\n' + uc._read("smc_mailbox.cuh")
    if proposal is not None:
        text += '\nnamespace bk_proposal {\n#line 1 "proposal.cu"\n' + proposal + "\n}  // namespace bk_proposal\n"
    text += '\n#line 1 "bk_user_kernels.cuh"\n' + uc._read("user_kernels.cuh")
    opts = ["-arch=sm_100a", "-std=c++17", f"-DBK_PROGRAM={PROGRAM_SMC_MOVES}", f"-DBK_DIMS={D}",
            f"-DBK_USER_FUSED_MAX_D={uc.FUSED_MAX_D}", "--ptxas-options=-v", "-DBK_PRIOR_LIK=1", "-DBK_SMC_KERNELS=1",
            f"-DBK_SMC_MAX_WORLD={uc.SMC_MAX_WORLD}", f"-DBK_SMC_MAILBOX_BYTES={uc.SMC_MAILBOX_BYTES}"]
    if f64:
        opts.append("--fmad=false")
    if proposal is not None:
        opts += [f"-DBK_PROPOSAL_NORMALS={normals}", f"-DBK_PROPOSAL_UNIFORMS={uniforms}",
                 f"-DBK_PROPOSAL_TRANSITION={transition}"]
    nv = uc.nvrtc()
    prog = C.c_void_p()
    assert nv.nvrtcCreateProgram(C.byref(prog), text.encode(), b"model.cu", 0, None, None) == 0
    arr = (C.c_char_p * len(opts))(*[o.encode() for o in opts])
    rc = nv.nvrtcCompileProgram(prog, len(opts), arr)
    n = C.c_size_t(0)
    nv.nvrtcGetProgramLogSize(prog, C.byref(n))
    buf = C.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(prog, buf)
    nv.nvrtcDestroyProgram(C.byref(prog))
    return rc == 0, buf.value.decode()


@uc.needs_nvrtc
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("D", [2, 16, 32])
def test_smc_moves_program_compiles(D, f64):
    ok, log = _compile_moves(D, f64, uc.PRIOR_LIK)
    assert ok, log
    assert uc.entries(log) == ["bk_user_smc_hmc_moves", "bk_user_smc_mala_moves", "bk_user_smc_rw_moves"]
    ok, log = _compile_moves(D, f64, uc.PRIOR_LIK, proposal=uc.WALK, normals=D, uniforms=0, transition=0)
    assert ok, log
    assert uc.entries(log) == ["bk_user_smc_mhp_moves"]


@uc.needs_nvrtc
@pytest.mark.parametrize("f64", [False, True])
def test_model_and_pair_programs_keep_their_entries(f64):
    ok, log = uc.compile_program(uc.PROGRAM_MODEL, 16, f64, model=uc.PRIOR_LIK, prior_lik=True)
    assert ok, log
    assert uc.entries(log) == sorted(["bk_user_eval", "bk_user_hmc", "bk_user_mala", "bk_user_mh", "bk_user_eval_pl",
                                      "bk_user_smc_rw", "bk_user_smc_mala", "bk_user_smc_hmc"])
    ok, log = uc.compile_program(uc.PROGRAM_MODEL_PROPOSAL, 16, f64, model=uc.PRIOR_LIK, proposal=uc.WALK,
                                 prior_lik=True, normals=16)
    assert ok, log
    assert uc.entries(log) == ["bk_user_mhp", "bk_user_smc_mhp"]
