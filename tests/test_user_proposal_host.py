"""bk_proposal_create_cuda without a GPU: argument validation and NVRTC compilation run before any device call; and the
proposal streams of oracle/proposals.py against device_rng.cuh itself, compiled for the host with nvcc."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from bayes_kit_b200 import _lib
from bayes_kit_b200.models import _load_nvrtc
from oracle import philox as ph
from oracle import proposals as opr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bayes-kit_b200", "csrc")

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


def _nvrtc_available():
    _load_nvrtc()
    try:
        C.CDLL("libnvrtc.so.12")
        return True
    except OSError:
        return False


needs_nvrtc = pytest.mark.skipif(not _nvrtc_available(), reason="NVRTC (libnvrtc.so.12) cannot be loaded")

DUMMY_PTR = 256   # never dereferenced: validation and compilation do not touch params


def _create(source, dims, dtype=_lib.BK_F32, params=DUMMY_PTR, n_params=1, normals=None, uniforms=0, transition=1,
            handle=True):
    h = _lib.u64(0)
    log = C.create_string_buffer(1 << 16)
    src = None if source is None else source.encode()
    rc = _lib.lib().bk_proposal_create_cuda(src, dims, dtype, params, n_params, dims if normals is None else normals,
                                            uniforms, transition, C.byref(h) if handle else None, log, len(log))
    if rc == _lib.BK_OK:
        assert h.value >> 62 == 1                  # proposal handles never equal a model handle
        assert _lib.lib().bk_proposal_destroy(h.value) == _lib.BK_OK
        assert _lib.lib().bk_proposal_destroy(h.value) == _lib.BK_E_HANDLE
    return rc, log.value.decode(), _lib.lib().bk_last_error().decode()


@needs_nvrtc
@pytest.mark.parametrize("kw,msg", [
    (dict(source=None, dims=2), "source"),
    (dict(source=RW, dims=2, handle=False), "handle_out"),
    (dict(source=RW, dims=0), "dims"),
    (dict(source=RW, dims=65537, normals=1), "dims"),
    (dict(source=RW, dims=2, dtype=7), "dtype"),
    (dict(source=RW, dims=2, params=None, n_params=1), "n_params"),
    (dict(source=RW, dims=2, params=DUMMY_PTR, n_params=0), "n_params"),
    (dict(source=RW, dims=2, params=DUMMY_PTR, n_params=-1), "n_params"),
    (dict(source=RW, dims=2, normals=-1), "n_normals"),
    (dict(source=RW, dims=2, normals=65537), "n_normals"),
    (dict(source=RW, dims=2, uniforms=-1), "n_uniforms"),
    (dict(source=RW, dims=2, uniforms=65), "n_uniforms"),
])
def test_arguments_rejected_before_compiling(kw, msg):
    rc, log, err = _create(**kw)
    assert rc == _lib.BK_E_INVALID
    assert msg in err
    assert log == ""


@needs_nvrtc
@pytest.mark.parametrize("source,transition,diag", [
    # diagnostics in the user's source carry its own line numbers
    ("\n\n__device__ void propose(const bk_real* t, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p)"
     " { q[0] = t[0] }", 0, "proposal.cu(3): error: expected a \";\""),
    ("__device__ void propos(const bk_real* t, bk_real* q, const bk_real* z, const bk_real* u, const bk_real* p) {}",
     0, "propose"),
    (RW.split("__device__ bk_real transition_log_density")[0], 1, "transition_log_density"),
])
def test_compile_error_returns_the_log(source, transition, diag):
    rc, log, err = _create(source, 3, transition=transition)
    assert rc == _lib.BK_E_INVALID
    assert diag in log and "error" in log
    assert "compilation failed" in err and "\n" not in err


@needs_nvrtc
def test_transition_is_optional_without_hastings():
    rc, log, err = _create(RW.split("__device__ bk_real transition_log_density")[0], 3, transition=0)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err


@needs_nvrtc
@pytest.mark.parametrize("dtype", [_lib.BK_F32, _lib.BK_F64])
@pytest.mark.parametrize("dims,normals,uniforms", [(2, None, 0), (17, 5, 3), (100, 101, 64)])
def test_valid_source_gets_past_compilation(dims, normals, uniforms, dtype):
    """BK_OK with a device, BK_E_CUDA (loading the module) without one -- never BK_E_INVALID."""
    rc, log, err = _create(RW, dims, dtype, normals=normals, uniforms=uniforms)
    assert rc in (_lib.BK_OK, _lib.BK_E_CUDA), err
    assert "bk_user_propose" in log                    # ptxas's resource report
    assert "bk_user_eval" not in log                   # a proposal program holds no model kernel


@needs_nvrtc
def test_proposal_handles_are_not_model_handles():
    assert _lib.lib().bk_mh_cuda_sample(1, 1, None, None, None, 1, 0, 1, None, None, None, 0, None) == _lib.BK_E_HANDLE
    assert _lib.lib().bk_mh_cuda_workspace_bytes(1, 1, 10) == 0


# ---- the proposal streams of oracle/proposals.py against device_rng.cuh -----------------------------------------------
_HOST_PROGRAM = r"""
#include <stdio.h>
#include <string.h>
#include "device_rng.cuh"
int main() {
    unsigned long long seed;
    int D, k;
    unsigned chain, draw;
    while (scanf("%llu %d %d %u %u", &seed, &D, &k, &chain, &draw) == 5) {
        const int b = bk::proposal_normal_block(k, D);
        uint32_t r[4];
        bk::Philox::gen(seed, (uint32_t)b, bk::TAG_NORMAL, chain, draw, r);
        float u = bk::philox_uniform<float>(seed, (uint32_t)k, chain, draw);
        double d = bk::philox_uniform<double>(seed, (uint32_t)k, chain, draw);
        uint32_t ub; unsigned long long db;
        memcpy(&ub, &u, 4); memcpy(&db, &d, 8);
        printf("%d %u %u %u %u %u %llu\n", b, r[0], r[1], r[2], r[3], ub, db);
    }
    return 0;
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand) and os.access(cand, os.X_OK):
            return cand
    return None


def test_proposal_streams_match_device_rng(tmp_path):
    """b(k) and the TAG_UNIFORM proposal uniforms, word for word: D = 1, 4, 5 and 17 with k past 4 ceil(D / 4), so the
    skipped accept block is crossed."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("no nvcc")
    src, exe = tmp_path / "prop_rng.cu", tmp_path / "prop_rng"
    src.write_text(_HOST_PROGRAM)
    r = subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", f"-I{CSRC}",
                        str(src), "-o", str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    rng = np.random.default_rng(7)
    rows = []
    for seed in (0, 42, 0xDEADBEEFCAFEF00D):
        for D in (1, 4, 5, 17):
            for k in range(4 * ph.accept_block(D) + 9):
                rows.append((seed, D, k, int(rng.integers(0, 2 ** 32)), int(rng.integers(0, 2 ** 32))))
    inp = "".join(" ".join(str(v) for v in row) + "\n" for row in rows)
    out = subprocess.run([str(exe)], input=inp, capture_output=True, text=True, timeout=60, check=True).stdout
    got = np.array([[int(v) for v in line.split()] for line in out.splitlines()], dtype=np.uint64)
    assert got.shape == (len(rows), 7)
    for i, (seed, D, k, chain, draw) in enumerate(rows):
        b = int(opr.proposal_normal_block(k, D))
        assert got[i, 0] == b and b != ph.accept_block(D)
        assert opr.proposal_blocks(D, k + 1)[k // 4] == b
        assert [int(w) for w in ph.gen(seed, b, ph.TAG_NORMAL, chain, draw)] == [int(v) for v in got[i, 1:5]]
        u = opr.proposal_uniforms(seed, chain, draw, 1, k + 1, np.float32)[0, k]
        d = opr.proposal_uniforms(seed, chain, draw, 1, k + 1, np.float64)[0, k]
        assert int(np.float32(u).view(np.uint32)) == int(got[i, 5])
        assert int(np.float64(d).view(np.uint64)) == int(got[i, 6])
    # with n_normals <= D the proposal reads exactly the random walk's blocks
    for D in (1, 4, 5, 17, 32):
        assert opr.proposal_blocks(D, D) == list(range(ph.accept_block(D)))
