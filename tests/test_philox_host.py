"""The NumPy restatement of the device random streams (oracle/philox.py), checked without a GPU: the Random123
known-answer vectors of Philox4x32-10, the uniform grids at their extremes, and -- when nvcc is installed -- the
host side of device_rng.cuh itself, word for word over a grid of counters and seeds."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import philox as ph

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bayes-kit_b200", "csrc")


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    got = ph.philox4x32_10(ctr, key)
    assert [int(w) for w in got] == list(want)


def test_gen_key_is_seed_low_high():
    seed = 0x299F31D0A4093822
    got = ph.gen(seed, 0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344)
    assert [int(w) for w in got] == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_vectorised_equals_scalar():
    rng = np.random.default_rng(0)
    c = rng.integers(0, 2 ** 32, size=(4, 50), dtype=np.uint64)
    k = rng.integers(0, 2 ** 32, size=(2, 50), dtype=np.uint64)
    vec = np.stack(ph.philox4x32_10(c, k))
    for i in range(50):
        one = ph.philox4x32_10(c[:, i], k[:, i])
        assert [int(w) for w in one] == [int(w) for w in vec[:, i]]


def test_uniform_grids_strictly_inside_unit_interval():
    lo, hi = ph.u01(0), ph.u01(0xFFFFFFFF)
    assert lo.dtype == np.float32 and 0.0 < lo and hi < 1.0
    assert lo == np.float32(2.0 ** -24) and hi == np.float32(1.0 - 2.0 ** -24)
    dlo, dhi = ph.u01d(0, 0), ph.u01d(0xFFFFFFFF, 0xFFFFFFFF)
    assert 0.0 < dlo and dhi < 1.0
    assert dlo == 2.0 ** -53 and dhi == 1.0 - 2.0 ** -53


def test_uniform_and_accept_word_selection():
    """philox_uniform<float>(k) is word k & 3 of block k >> 2; <double>(k) the word pair k & 1 of block k >> 1;
    the accept uniform is word 0 (pair 0, 1) of block ceil(D / 4) of the normal stream."""
    seed, chain, draw = 0x123456789ABCDEF, 7, 3
    for k in range(12):
        r = ph.gen(seed, k >> 2, ph.TAG_UNIFORM, chain, draw)
        assert ph.philox_uniform(seed, k, chain, draw) == ph.u01(r[k & 3])
        r = ph.gen(seed, k >> 1, ph.TAG_UNIFORM, chain, draw)
        want = ph.u01d(r[2], r[3]) if k & 1 else ph.u01d(r[0], r[1])
        assert ph.philox_uniform(seed, k, chain, draw, np.float64) == want
    for D, blk in ((1, 1), (4, 1), (5, 2), (100, 25), (101, 26)):
        assert ph.accept_block(D) == blk
        r = ph.gen(seed, blk, ph.TAG_NORMAL, chain, draw)
        assert ph.accept_uniform(seed, chain, draw, D) == ph.u01(r[0])
        assert ph.accept_uniform(seed, chain, draw, D, np.float64) == ph.u01d(r[0], r[1])


def test_normals_layout_and_moments():
    """init_normal: element e is word e % 4 of block e // 4; both Box-Muller forms are standard normal and agree
    with each other in distribution (not value: they read different words)."""
    z = ph.init_normal(5, 3, 0, 7, 10)
    blk = ph.normal4_f64(5, 2, 3 + 4, 0)
    np.testing.assert_array_equal(z[4, 8:10], blk[:2])
    for dt in (np.float64, np.float32):
        z = ph.init_normal(11, 0, 2, 4000, 16, dt).ravel()
        assert abs(z.mean()) < 5 / np.sqrt(z.size) and abs(z.var() - 1) < 5 * np.sqrt(2 / z.size)
        assert np.abs(z).max() < 7


def test_sincospi_reduction():
    x = np.linspace(1e-6, 2 - 1e-6, 10001)
    s, c = ph._sincospi(x)
    np.testing.assert_allclose(s, np.sin(np.pi * x), atol=1e-15)
    np.testing.assert_allclose(c, np.cos(np.pi * x), atol=1e-15)


_HOST_PROGRAM = r"""
#include <stdio.h>
#include <string.h>
#include "device_rng.cuh"
int main() {
    unsigned long long seed;
    unsigned block, tag, chain, draw;
    while (scanf("%llu %u %u %u %u", &seed, &block, &tag, &chain, &draw) == 5) {
        uint32_t r[4];
        bk::Philox::gen(seed, block, tag, chain, draw, r);
        float u = bk::u01(r[0]);
        double d = bk::u01d(r[0], r[1]);
        uint32_t ub; unsigned long long db;
        memcpy(&ub, &u, 4); memcpy(&db, &d, 8);
        printf("%u %u %u %u %u %llu\n", r[0], r[1], r[2], r[3], ub, db);
    }
    return 0;
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand) and os.access(cand, os.X_OK):
            return cand
    return None


def test_device_rng_header_matches_restatement(tmp_path):
    """Philox::gen, u01 and u01d are __host__ __device__: a host program compiled against device_rng.cuh must
    produce the restatement's words and uniforms bit for bit."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("no nvcc")
    src, exe = tmp_path / "rng.cu", tmp_path / "rng"
    src.write_text(_HOST_PROGRAM)
    r = subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", f"-I{CSRC}",
                        str(src), "-o", str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    rng = np.random.default_rng(1)
    rows = [(0, 0, 0, 0, 0), (2 ** 64 - 1, 2 ** 32 - 1, 3, 2 ** 32 - 1, 2 ** 32 - 1)]
    for seed in (0, 1, 42, 0xDEADBEEFCAFEF00D, 2 ** 63 + 5):
        for _ in range(40):
            rows.append((seed, int(rng.integers(0, 300)), int(rng.integers(0, 4)), int(rng.integers(0, 2 ** 32)),
                         int(rng.integers(0, 2 ** 32))))
    inp = "".join(" ".join(str(v) for v in row) + "\n" for row in rows)
    out = subprocess.run([str(exe)], input=inp, capture_output=True, text=True, timeout=60, check=True).stdout
    got = np.array([[int(v) for v in line.split()] for line in out.splitlines()], dtype=np.uint64)
    assert got.shape == (len(rows), 6)
    a = np.array(rows, dtype=np.uint64).T
    words = np.stack(ph.gen(a[0], a[1], a[2], a[3], a[4]), 1).astype(np.uint64)
    np.testing.assert_array_equal(got[:, :4], words)
    u = ph.u01(words[:, 0].astype(np.uint32)).view(np.uint32).astype(np.uint64)
    d = ph.u01d(words[:, 0].astype(np.uint32), words[:, 1].astype(np.uint32)).view(np.uint64)
    np.testing.assert_array_equal(got[:, 4], u)
    np.testing.assert_array_equal(got[:, 5], d)
