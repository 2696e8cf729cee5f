"""The transform-size and pass-plan rules of fft_autocorr.cu, checked without a GPU: a host program compiled from
the translation unit itself prints rfft_size / rfft_plan / fft_size / fft_plan, and tests/_diag_plans.py (the
restatement the GPU tests choose their lengths with) must agree line for line.  Also pins the coverage facts the GPU
tests rely on: 37 half-lengths, the radix-3 plans and the (16, 2), (2, 1) tails."""
import os
import shutil
import subprocess

import pytest

import _diag_plans as dp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bayes-kit_b200", "csrc")

_HOST_PROGRAM = r"""
#include <stdio.h>
#include "fft_autocorr.cu"
namespace bk {           // the two library symbols the translation unit refers to (core.cu)
std::atomic<uint64_t> g_launches{0};
void set_error(const char*, ...) {}
}
int main() {
    long long N;
    while (scanf("%lld", &N) == 1) {
        const long long S = (long long)bk::rfft_size(N);
        printf("%lld rfft %lld", N, S);
        if (S) {
            const bk::RfftPlan p = bk::rfft_plan((int)(S / 2));
            printf(" %d", p.M);
            for (int i = 0; i < p.n_pass; ++i) printf(" %d:%d", p.radix[i], p.m[i]);
        }
        const long long F = (long long)bk::fft_size(N);
        const bk::FftPlan f = bk::fft_plan(F);
        printf(" fft %lld %d", F, f.log2S);
        for (int i = 0; i < f.n_pass; ++i) printf(" %d", f.log2r[i]);
        printf("\n");
    }
    return 0;
}
"""

LARGE_N = (10241, 10242, 16384, 16385, 32768, 32769, 65536, 65537, 131072, 131073, 262144, 262145, 524288, 524289)


def _expected_line(N):
    S = dp.rfft_size(N)
    words = [str(N), "rfft", str(S)]
    if S:
        words.append(str(S // 2))
        words += [f"{r}:{m}" for r, m in dp.rfft_plan(S // 2)]
    F = dp.fft_size(N)
    words += ["fft", str(F), str(F.bit_length() - 1)] + [str(r) for r in dp.fft_plan(F)]
    return " ".join(words)


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand) and os.access(cand, os.X_OK):
            return cand
    return None


def test_plan_rules_match_fft_autocorr(tmp_path):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("no nvcc")
    src, exe = tmp_path / "plans.cu", tmp_path / "plans"
    src.write_text(_HOST_PROGRAM)
    r = subprocess.run([nvcc, "-std=c++17", "--expt-relaxed-constexpr", "-gencode", "arch=compute_100a,code=sm_100a",
                        f"-I{CSRC}", str(src), "-o", str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    ns = list(range(2, 10242)) + list(LARGE_N)
    out = subprocess.run([str(exe)], input="".join(f"{n}\n" for n in ns), capture_output=True, text=True,
                         timeout=120, check=True).stdout.splitlines()
    assert len(out) == len(ns)
    bad = [(got, _expected_line(n)) for n, got in zip(ns, out) if got.strip() != _expected_line(n)]
    assert not bad, bad[:5]


def test_plan_coverage_facts():
    by_m = dp.rfft_lengths()
    # 37 half-lengths M = c 2^a (c in {1, 3, 5}), the largest 10,240; beyond N = 10,240 the global transform
    assert len(by_m) == 37 and max(by_m) == 10240
    assert dp.rfft_size(10240) == 20480 and dp.rfft_size(10241) == 0
    for M in by_m:
        c = M
        while c % 2 == 0:
            c //= 2
        assert c in (1, 3, 5)
        assert by_m[M] == list(range(by_m[M][0], by_m[M][-1] + 1))    # each M serves one run of N
    assert by_m[1536] == list(range(1281, 1537))
    # radix 3 leads every plan with a factor 3, and is followed by radix-16 passes from M = 96 on
    radix3 = sorted(M for M in by_m if any(r == 3 for r, _ in dp.rfft_plan(M)))
    assert radix3 == [3, 6, 12, 24, 48, 96, 192, 384, 768, 1536, 3072, 6144]
    for M in radix3:
        assert dp.rfft_plan(M)[0] == (3, M // 3)
    assert dp.rfft_plan(1536) == ((3, 512), (16, 32), (16, 2), (2, 1))
    # the (16, m = 2), (2, 1) tail
    tails = sorted(M for M in by_m if dp.rfft_plan(M)[-2:] == ((16, 2), (2, 1)))
    assert tails == [32, 96, 160, 512, 1536, 2560, 8192]
    # both addressing modes of rf_pass occur, and the non-linear one only for m < 8 with R m > 8
    passes = set().union(*(dp.rfft_passes(M) for M in by_m))
    assert {lin for _, _, lin in passes} == {True, False}
    assert all(m < 8 and r * m > 8 for r, m, lin in passes if not lin)
    # the global transform: radix-32 passes, the remainder last; S = 2^20 is four full passes
    assert dp.fft_plan(1 << 20) == (5, 5, 5, 5) and dp.fft_plan(1 << 16) == (5, 5, 5, 1)
    assert dp.fft_size(524288) == 1 << 20 and dp.fft_size(524289) == 1 << 21
    # k_ess_stream's regimes
    assert dp.ess_regime(30, 10_000) == "first-pass" and dp.ess_regime(32, 10_000) == "multi-pass"
    assert dp.ess_regime(767, 10_000) == "multi-pass" and dp.ess_regime(768, 10_000) == "far-lag"
