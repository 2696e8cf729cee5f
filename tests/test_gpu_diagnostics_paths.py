"""autocorr, iat and ess against the fp64 NumPy reference (oracle/diagnostics.py) on every path the device kernels
can choose: every half-length and pass of the shared-memory real FFT (k_acf_rfft), every pass split of the
global-scratch transform (k_acf_fft) up to S = 2^20, the direct sums (k_acf_direct), and the streaming Geyer
kernel (k_ess_stream) in its first-pass, multi-pass and far-lag regimes, through the 16-byte and element-wise fp32
staging, fp64, strided series, and gathered chunks of strided series.  Same array in, 1e-9 out (BASELINE); fp32
input is compared on the array cast to fp64.

The Geyer truncation is discontinuous: a pair sum within rounding of zero may stop the sum one pair earlier or later
on the device.  Series with such a pair (|pair| < 1e-12 up to the truncation point) are left out of the 1e-9 check
and counted; every other series is checked strictly.  Likewise ess = N / iat is not compared where iat = 2 sum - 1
cancels to rounding level (|iat| < 1e-6, e.g. acor_1 = -1/2 at N = 4): iat itself is still held to 1e-10 there.
The k_ess_stream regimes (first pass only, multi-pass, far-lag) each test reaches are asserted from the oracle's
truncation points."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.signal import lfilter

import _diag_plans as dp
from _dev import np_
from oracle import diagnostics as od

pytestmark = pytest.mark.gpu
TOL = dict(rtol=1e-9, atol=1e-10)
TIE = 1e-12
IAT_MIN = 1e-6
PHIS = (-0.9, -0.5, 0.0, 0.5, 0.9, 0.99, 0.998)

# every pass rf_pass_r can run: (radix, m = block length after the pass, linear addressing of the skewed line)
RFFT_PASSES = {(2, 1, True), (3, 1, True), (3, 2, True), (3, 4, False), (3, 8, True), (3, 16, True), (3, 32, True),
               (3, 64, True), (3, 128, True), (3, 256, True), (3, 512, True), (3, 1024, True), (3, 2048, True),
               (4, 1, True), (5, 1, True), (5, 2, False), (5, 4, False), (5, 8, True), (5, 16, True), (5, 32, True),
               (5, 64, True), (5, 128, True), (5, 256, True), (5, 512, True), (5, 1024, True), (5, 2048, True),
               (8, 1, True), (16, 1, False), (16, 2, False), (16, 4, False), (16, 8, True), (16, 16, True),
               (16, 32, True), (16, 64, True), (16, 128, True), (16, 256, True), (16, 512, True)}
# every pass split of the global transform (log2 of each pass's radix), S = 2^2 .. 2^20
FFT_SPLITS = {(2,), (3,), (4,), (5,), (5, 1), (5, 2), (5, 3), (5, 4), (5, 5), (5, 5, 1), (5, 5, 2), (5, 5, 3),
              (5, 5, 4), (5, 5, 5), (5, 5, 5, 1), (5, 5, 5, 2), (5, 5, 5, 3), (5, 5, 5, 4), (5, 5, 5, 5)}


def _rfft_ns():
    ns = set(range(2, 17))
    for lst in dp.rfft_lengths().values():
        ns |= {lst[0], lst[-1]}
    return sorted(ns)


RFFT_NS = _rfft_ns()
FFT_PRODUCTION_NS = (10241, 16385, 65536, 65537, 262144, 524288)
FFT_FORCED_NS = sorted({n for k in range(1, 14) for n in (2 ** k, 2 ** k + 1)})

# the chosen lengths reach every pass and every split before anything runs on the device
assert {dp.rfft_size(n) // 2 for n in RFFT_NS} == set(dp.rfft_lengths())
assert set().union(*(dp.rfft_passes(dp.rfft_size(n) // 2) for n in RFFT_NS)) == RFFT_PASSES
assert {n for n in RFFT_NS if dp.rfft_size(n) // 2 == 1536} == {1281, 1536}
assert all(dp.rfft_size(n) == 0 for n in FFT_PRODUCTION_NS)
assert {dp.fft_plan(dp.fft_size(n)) for n in FFT_PRODUCTION_NS + tuple(FFT_FORCED_NS)} == FFT_SPLITS

ERR, TIES, SEEN, DEGENERATE = {}, {}, {}, {}


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for k in sorted(ERR):
        print(f"\n[diagnostics paths] {k}: largest error {ERR[k]:.3g} over {SEEN[k]} values"
              f"{f', {TIES[k]} near-tie series left out' if k in TIES else ''}"
              f"{f', {DEGENERATE[k]} ess values with |iat| < {IAT_MIN:g} left out' if k in DEGENERATE else ''}")


def _close(path, got, want, rel):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    np.testing.assert_allclose(got, want, err_msg=path, **TOL)
    d = np.abs(got - want)
    e = float((d / np.abs(want)).max() if rel else d.max()) if d.size else 0.0
    ERR[path] = max(ERR.get(path, 0.0), e)
    SEEN[path] = SEEN.get(path, 0) + d.size


def ar1(phi, s, n, rng):
    """[s, n] AR(1) rows, x_t = phi x_{t-1} + e_t (od.sample_ar1 vectorised)."""
    return lfilter([1.0], [1.0, -phi], rng.normal(size=(s, n)), axis=1)


def dev(rows, dtype, draws_first):
    """[S, N] host rows -> device tensor in the layout (draws_first: [N, S])."""
    t = torch.as_tensor(rows, dtype=dtype, device="cuda")
    return t.t().contiguous() if draws_first else t.contiguous()


def seen_rows(x, draws_first):
    """The fp64 [S, N] rows the device reads from x."""
    r = np_(x).astype(np.float64)
    return np.ascontiguousarray(r.T if draws_first else r)


# =============================================================================== autocorr
def _acf(bk, path, rows, dtype, draws_first):
    x = dev(rows, dtype, draws_first)
    got = np_(bk.autocorr(x, draws_first=draws_first))
    _close(path, got, od.autocorr_batch(seen_rows(x, draws_first)), rel=False)


def test_autocorr_rfft_every_half_length(bk, monkeypatch):
    """k_acf_rfft: the smallest and largest N of each of the 37 half-lengths, and N = 2..16; fp64 / fp32, odd and
    even series counts, contiguous and draws_first."""
    monkeypatch.setenv("BK_ACF", "fft")
    monkeypatch.delenv("BK_ACF_RFFT", raising=False)
    rng = np.random.default_rng(10)
    for i, n in enumerate(RFFT_NS):
        d1, d2 = (torch.float64, torch.float32) if i % 2 == 0 else (torch.float32, torch.float64)
        _acf(bk, "autocorr rfft", 2.5 + ar1(0.7, 3, n, rng), d1, False)
        _acf(bk, "autocorr rfft", -1.0 + ar1(-0.4, 2, n, rng), d2, True)


def test_autocorr_rfft_grid_stride(bk, monkeypatch):
    """More series than k_acf_rfft's persistent grid (sms x 2 CTAs at M = 1536): every series compared."""
    monkeypatch.setenv("BK_ACF", "fft")
    monkeypatch.delenv("BK_ACF_RFFT", raising=False)
    rng = np.random.default_rng(11)
    _acf(bk, "autocorr rfft", ar1(0.9, 301, 1536, rng), torch.float64, False)
    _acf(bk, "autocorr rfft", 4.0 + ar1(0.3, 301, 1281, rng), torch.float32, True)


def test_autocorr_global_fft_production_sizes(bk, monkeypatch):
    """k_acf_fft beyond the on-chip limit, S = 2^15 .. 2^20; 1, 2 and 3 series (a pair left incomplete)."""
    monkeypatch.delenv("BK_ACF", raising=False)
    monkeypatch.delenv("BK_ACF_RFFT", raising=False)
    rng = np.random.default_rng(12)
    for n in FFT_PRODUCTION_NS:
        _acf(bk, "autocorr global fft", 1.5 + ar1(0.8, 1, n, rng), torch.float64, False)
        _acf(bk, "autocorr global fft", ar1(0.5, 2, n, rng), torch.float32, True)
        _acf(bk, "autocorr global fft", -3.0 + ar1(0.95, 3, n, rng), torch.float64, True)
        _acf(bk, "autocorr global fft", ar1(-0.6, 3, n, rng), torch.float32, False)


def test_autocorr_global_fft_second_pair_per_cta(bk, monkeypatch):
    """299 series = 150 pairs on at most 148 CTAs: two CTAs transform a second pair, the last one incomplete."""
    monkeypatch.delenv("BK_ACF", raising=False)
    monkeypatch.delenv("BK_ACF_RFFT", raising=False)
    rng = np.random.default_rng(13)
    _acf(bk, "autocorr global fft", 2.0 + ar1(0.6, 299, 10241, rng), torch.float64, False)
    _acf(bk, "autocorr global fft", ar1(0.9, 299, 10241, rng), torch.float32, True)


def test_autocorr_global_fft_every_split(bk, monkeypatch):
    """BK_ACF_RFFT=0: N = 2^k and 2^k + 1, k = 1..13 -> S = 4 .. 32768 through the global transform."""
    monkeypatch.setenv("BK_ACF", "fft")
    monkeypatch.setenv("BK_ACF_RFFT", "0")
    rng = np.random.default_rng(14)
    for i, n in enumerate(FFT_FORCED_NS):
        _acf(bk, "autocorr global fft", 0.5 + ar1(0.7, 3, n, rng), (torch.float64, torch.float32)[i % 2], bool(i % 3 == 0))
        _acf(bk, "autocorr global fft", ar1(-0.3, 2, n, rng), (torch.float32, torch.float64)[i % 2], True)


def test_autocorr_beyond_2_20_raises(bk, monkeypatch):
    monkeypatch.delenv("BK_ACF", raising=False)
    monkeypatch.delenv("BK_ACF_RFFT", raising=False)
    x = torch.zeros(524289, dtype=torch.float32, device="cuda")
    x[::2] = 1.0
    with pytest.raises(NotImplementedError, match=r"2\^20"):
        bk.autocorr(x)


def test_autocorr_direct_every_short_length(bk, monkeypatch):
    """k_acf_direct (the default for N <= 256): every N = 2..256, contiguous and strided; then more series than its
    1,184-block grid."""
    monkeypatch.delenv("BK_ACF", raising=False)
    rng = np.random.default_rng(15)
    for n in range(2, 257):
        _acf(bk, "autocorr direct", 1.0 + ar1(0.8, 3, n, rng), (torch.float64, torch.float32)[n % 2], False)
        _acf(bk, "autocorr direct", ar1(-0.5, 2, n, rng), (torch.float32, torch.float64)[n % 2], True)
    _acf(bk, "autocorr direct", ar1(0.5, 1200, 100, rng), torch.float64, False)


# =============================================================================== iat / ess
def oracle_geyer(rows):
    """Per row: iat_ipse, iat_imse, the truncation point (end_pos_pairs) and whether a pair sum up to it lies within
    TIE of zero."""
    out = np.empty((len(rows), 4))
    for i, r in enumerate(rows):
        ac = od.autocorr(r)
        e = od.end_pos_pairs(ac)
        npr = len(ac) // 2
        pairs = (ac[0:2 * npr:2] + ac[1:2 * npr:2])[:e // 2 + 1]
        out[i] = od.iat_ipse(r), od.iat_imse(r), e, float(np.any(np.abs(pairs) < TIE))
    return out


def iat_ess(x, draws_first=False, ws_bytes=None):
    """bk_iat_ess through the C ABI, both estimators -> {"ipse": (iat, ess), "imse": (iat, ess)}; ws_bytes
    overrides the workspace the library asks for (it sets how many gathered series fit per chunk)."""
    from bayes_kit_b200 import _lib as L
    from bayes_kit_b200._diag import as_series
    xt, _, lay = as_series(x, draws_first=draws_first)
    assert xt.data_ptr() == x.data_ptr()
    lib = L.lib()
    dt = L.BK_F32 if x.dtype == torch.float32 else L.BK_F64
    if ws_bytes is None:
        ws_bytes = lib.bk_iat_ess_workspace_bytes(dt, C.byref(lay))
    ws = torch.empty(max(int(ws_bytes), 1), dtype=torch.uint8, device="cuda")
    res = {}
    for name, est in (("ipse", L.IAT_IPSE), ("imse", L.IAT_IMSE)):
        t = torch.full((lay.n_series,), float("nan"), dtype=torch.float64, device="cuda")
        e = torch.full_like(t, float("nan"))
        L.check(lib.bk_iat_ess(x.data_ptr(), dt, C.byref(lay), est, t.data_ptr(), e.data_ptr(),
                               ws.data_ptr() if ws_bytes else None, ws_bytes, torch.cuda.current_stream().cuda_stream))
        res[name] = (np_(t), np_(e))
    return res


def check_geyer(path, got, want, n, idx=None):
    """got: iat_ess() of the whole array; want: oracle_geyer() of rows idx (all when None).  Returns the regimes."""
    idx = np.arange(len(want)) if idx is None else np.asarray(idx)
    keep = want[:, 3] == 0
    TIES[path] = TIES.get(path, 0) + int((~keep).sum())
    assert (~keep).sum() <= max(2, len(want) // 100), f"{path}: {(~keep).sum()} near-tie series of {len(want)}"
    for j, name in enumerate(("ipse", "imse")):
        t, e = got[name]
        _close(path, t[idx][keep], want[keep, j], rel=False)
        # ess = N / iat: where iat = 2 sum - 1 cancels to rounding level (|iat| < IAT_MIN, e.g. acor_1 = -1/2 at
        # N = 4) both sides divide by noise; iat itself is still held to the absolute tolerance above
        ok = keep & (np.abs(want[:, j]) >= IAT_MIN)
        DEGENERATE[path] = DEGENERATE.get(path, 0) + int((keep & ~ok).sum())
        assert (keep & ~ok).sum() <= max(3, len(want) // 100), f"{path}: {(keep & ~ok).sum()} series with iat ~ 0"
        _close(path, e[idx][ok], n / want[ok, j], rel=True)
    return {dp.ess_regime(int(ep), n) for ep in want[:, 2]}


def ess_kinds(n, rng):
    """[9, n]: AR(1) at every phi in PHIS, 1e4 + AR(1) (fp32-representable: exercises the provisional centre), and
    a chain with runs of repeated values (rejected proposals)."""
    rows = [ar1(phi, 1, n, rng)[0] for phi in PHIS]
    rows.append((1e4 + ar1(0.9, 1, n, rng)[0]).astype(np.float32).astype(np.float64))
    rep = ar1(0.5, 1, n, rng)[0]
    src, t = np.empty(n), 0
    for run in range(n):                       # runs of length 1, 2, 3, 4, 1, ...
        ln = 1 + run % 4
        src[t:t + ln] = rep[run]
        t += ln
        if t >= n:
            break
    rows.append(src)
    return np.stack(rows)


ESS_NS = list(range(4, 41)) + [255, 256, 257, 767, 768, 769, 1023, 1024]


def test_ess_stream_lengths_and_layouts(bk):
    """k_ess_stream at N = 4..40 (lanes beyond N in the head / tail correction), the chunk and ring edges, every
    N % 4: fp64, fp32 rows (all 16-byte aligned when N % 4 == 0, a mix otherwise), and draws_first with fewer than
    64 series (strided, element-wise staging)."""
    assert {n % 4 for n in ESS_NS} == {0, 1, 2, 3}
    rng = np.random.default_rng(20)
    regimes = set()
    for n in ESS_NS:
        rows = ess_kinds(n, rng)
        want64 = oracle_geyer(rows)
        want32 = oracle_geyer(rows.astype(np.float32).astype(np.float64))
        f32 = "stream fp32 vec" if n % 4 == 0 else "stream fp32 vec + element"
        regimes |= check_geyer("stream fp64", iat_ess(dev(rows, torch.float64, False)), want64, n)
        regimes |= check_geyer(f32, iat_ess(dev(rows, torch.float32, False)), want32, n)
        regimes |= check_geyer("stream fp32 element (strided)", iat_ess(dev(rows, torch.float32, True), True),
                               want32, n)
        regimes |= check_geyer("stream fp64 (strided)", iat_ess(dev(rows, torch.float64, True), True), want64, n)
    assert regimes >= {"first-pass", "multi-pass"}


def test_ess_stream_misaligned_fp32(bk):
    """A 1-D fp32 view at storage offset 1, 2, 3: contiguous, so passed through as is, but not 16-byte aligned."""
    rng = np.random.default_rng(21)
    for n in (5, 37, 256, 257, 1023, 1024, 4099):
        rows = ess_kinds(n, rng)[[3, 5, 7, 8]].astype(np.float32)
        want = oracle_geyer(rows.astype(np.float64))
        for off in (1, 2, 3):
            for i, r in enumerate(rows):
                base = torch.zeros(n + 4, dtype=torch.float32, device="cuda")
                base[off:off + n] = torch.as_tensor(r, device="cuda")
                x = base[off:off + n]
                assert x.is_contiguous() and x.data_ptr() % 16 != 0
                check_geyer("stream fp32 element (misaligned)", iat_ess(x), want[i:i + 1], n)


def test_ess_stream_far_lag(bk):
    """phi = 0.998 over ~200k draws: the truncation lies beyond lag 768, where k_ess_stream leaves the shared-memory
    ring for plain strided sums; phi = 0.95 truncates in the multi-pass range."""
    rng = np.random.default_rng(22)
    n = 200_003
    rows = np.concatenate([ar1(0.998, 3, n, rng), 7.0 + ar1(0.95, 2, n, rng)])
    for dtype, df, path in ((torch.float64, False, "stream fp64"), (torch.float32, False, "stream fp32 vec + element"),
                            (torch.float32, True, "stream fp32 element (strided)")):
        x = dev(rows, dtype, df)
        want = oracle_geyer(seen_rows(x, df))
        ends = want[:, 2]
        assert (ends[:3] >= 768).any() and ((ends >= 32) & (ends < 736)).any(), ends
        assert check_geyer(path, iat_ess(x, df), want, n) >= {"multi-pass", "far-lag"}


def _mixed_rows(s, n, rng):
    kinds = [ess_kinds(n, rng) for _ in range((s + 8) // 9)]
    return np.concatenate(kinds)[:s]


@pytest.mark.parametrize("n", [256, 257])
def test_ess_gather_every_chunk(bk, n):
    """draws_first with >= 64 series: strided series gathered into scratch chunk by chunk.  Workspaces that fit 32,
    33 (rounded down to 32) and 100 (-> 96) series: several chunks and a ragged last one; every series compared."""
    rng = np.random.default_rng(23 + n)
    rows = _mixed_rows(230, n, rng)
    for dtype, esz in ((torch.float32, 4), (torch.float64, 8)):
        x = dev(rows, dtype, True)
        want = oracle_geyer(seen_rows(x, True))
        for fit in (32, 33, 100, None):
            ws = None if fit is None else 256 + fit * n * esz
            check_geyer("gather", iat_ess(x, True, ws), want, n)


def test_ess_stream_grid_stride(bk):
    """More series than k_ess_stream's grid (296 blocks x 8 warps = 2,368): every series compared."""
    rng = np.random.default_rng(24)
    for s, n, dtype in ((2500, 64, torch.float32), (2400, 37, torch.float64)):
        x = dev(_mixed_rows(s, n, rng), dtype, False)
        check_geyer("stream fp32 vec" if dtype == torch.float32 else "stream fp64", iat_ess(x),
                    oracle_geyer(seen_rows(x, False)), n)


def test_ess_bench_shape_in_miniature(bk):
    """The benchmark's min_ess_per_s shape in miniature: fp32 draws_first, N = 200, 65,536 + 32 series through the
    library's own workspace (a full 65,536-series chunk and a ragged one); a subset spread over both compared."""
    rng = np.random.default_rng(25)
    s, n = 65536 + 32, 200
    rows = np.concatenate([ar1(phi, s // len(PHIS) + 1, n, rng) for phi in PHIS])[:s]
    rows = rows[rng.permutation(s)]
    x = dev(rows, torch.float32, True)
    idx = np.unique(np.concatenate([np.arange(0, s, 61), np.arange(65536 - 40, s)]))
    got = iat_ess(x, True)
    check_geyer("gather", got, oracle_geyer(seen_rows(x, True)[idx]), n, idx)


def test_ess_block_kernel(bk, monkeypatch):
    """BK_ESS=block (k_acf_direct, whole series in shared memory) up to its limit of 25,584 draws."""
    monkeypatch.setenv("BK_ESS", "block")
    rng = np.random.default_rng(26)
    for n in (4, 5, 37, 257, 1024, 10_000, 25_584):
        rows = ess_kinds(n, rng)
        for dtype, df in ((torch.float64, False), (torch.float32, True)):
            x = dev(rows, dtype, df)
            check_geyer("block", iat_ess(x, df), oracle_geyer(seen_rows(x, df)), n)
    with pytest.raises(NotImplementedError):
        bk.ess(torch.ones(25_585, dtype=torch.float64, device="cuda"))


def test_ess_long_strided_series(bk):
    """fp32 draws_first, N = 2^21 + 64 draws x 64 series: more 32-draw tiles (65,538) than a grid's y extent."""
    rng = np.random.default_rng(27)
    n, s = 2 ** 21 + 64, 64
    rows = rng.standard_normal((s, n), dtype=np.float32)
    for i in (0, 31, 63):
        rows[i] = lfilter([1.0], [1.0, -0.5], rows[i].astype(np.float64))
    x = dev(rows, torch.float32, True)
    del rows
    got = np_(bk.ess(x, draws_first=True))
    assert got.shape == (s,) and np.isfinite(got).all()
    for i in (0, 31, 63):
        r = np_(x[:, i]).astype(np.float64)
        _close("gather", got[i], od.ess(r), rel=True)
