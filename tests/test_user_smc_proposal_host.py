"""The SMC's proposal move (proposal_kernel) without a GPU: the bk_smc_kernel layout the ctypes binding assumes, the
handle checks of its entry points, and the NumPy restatement of the move against the reference's recorded runs.
(Model and proposal handles cannot be created without a device: creation loads the compiled module.)"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import _smc_proposal_oracle as sop
from bayes_kit_b200 import _lib
from conftest import golden
from oracle import samplers as osm
from oracle.models import build_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_LAYOUT = r"""
#include <stddef.h>
#include <stdio.h>
#include "bk.h"
int main() {
    printf("%zu %zu %zu %zu %zu %d %d\n", sizeof(bk_smc_kernel), offsetof(bk_smc_kernel, kind),
           offsetof(bk_smc_kernel, steps), offsetof(bk_smc_kernel, scale), offsetof(bk_smc_kernel, proposal),
           (int)BK_SMC_KERNEL_PROPOSAL, (int)BK_SMC_PROPOSAL_MAX_NORMALS);
    return 0;
}
"""


def _compiler():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand) and os.access(cand, os.X_OK):
            return cand
    return None


def test_smc_kernel_layout_matches_bk_h(tmp_path):
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
    assert got == [C.sizeof(K), K.kind.offset, K.steps.offset, K.scale.offset, K.proposal.offset,
                   _lib.SMC_KERNEL_PROPOSAL, _lib.SMC_PROPOSAL_MAX_NORMALS]
    # the descriptors of the existing kinds leave the proposal at 0
    assert _lib.SmcKernel(_lib.SMC_KERNEL_RW, 0, 0.2).proposal == 0


def test_unknown_handles_are_refused_before_any_device_call():
    lib = _lib.lib()
    log = C.create_string_buffer(256)
    log.value = b"stale"
    assert lib.bk_smc_cuda_prepare(12345, 1 << 62, log, len(log)) == _lib.BK_E_HANDLE
    assert log.value == b""
    assert lib.bk_smc_cuda_prepare(0, 0, None, 0) == _lib.BK_E_HANDLE
    kn = _lib.SmcKernel(_lib.SMC_KERNEL_PROPOSAL, 0, 0.0, 1 << 62)
    sh, rng = _lib.SmcShard(), _lib.Rng()
    assert lib.bk_smc_shard_move(12345, C.byref(sh), None, 1, 1, C.byref(kn), C.byref(rng), 0, None, None, 0,
                                 None) == _lib.BK_E_HANDLE
    assert lib.bk_smc_shard_run(12345, C.byref(sh), None, 1, 1, 1, C.byref(kn), C.byref(rng), 0, 0.0, None, None,
                                None, 0, None) == _lib.BK_E_HANDLE


@pytest.mark.parametrize("name", ["smc_gauss_d5", "smc_gauss_d50", "smc_binom"])
def test_oracle_walk_restated_reproduces_the_rw_goldens(name):
    """The proposal move with the random walk restated is the reference's metropolis_kernel: the recorded indices
    exactly, and the same particles as oracle.samplers.smc_tempered's ("rw", s) kind, bit for bit."""
    z = golden(name)
    model, s, T = build_model(z), float(z["scale"]), int(z["T"])
    walk = lambda th, zz, u: th + s * zz
    th, idx, acc = sop.smc_tempered(model, z["thetas0"], z["normals"], z["acc_uniforms"], z["res_uniforms"], T, walk)
    assert np.array_equal(idx, z["indices"])
    np.testing.assert_allclose(th, z["thetas_final"], rtol=1e-12, atol=1e-14)
    rw, rw_idx = osm.smc_tempered(model, z["thetas0"], z["normals"], z["acc_uniforms"], z["res_uniforms"], s, T)
    assert np.array_equal(th, rw) and np.array_equal(idx, rw_idx)
    assert 0 < acc.mean() < 1
    # [T, M, 1] accept uniforms (a proposal without uniforms, the column layout) give the same run
    th1, idx1, _ = sop.smc_tempered(model, z["thetas0"], z["normals"], z["acc_uniforms"][..., None],
                                    z["res_uniforms"], T, walk)
    assert np.array_equal(th1, th) and np.array_equal(idx1, idx)
