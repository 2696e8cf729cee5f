"""fp32 kernels draw by draw against the fp64 oracle, in every lane layout.

The timed samplers run in fp32, and much of their code exists only there: the isotropic HMC position form
(x_{n+1} = c x_n - x_{n-1}), the wide 4x4 / 8x4 and narrow 4x5..4x7 lane layouts, the SMC move in the 4x4 / 8x2
layouts and the accept uniform taken from the spare normal block.  Moment tests do not resolve a wrong lane, a
padding slot in a sum or a slightly wrong energy; per-draw parity under injected streams does.

Tolerances (fp32 unit roundoff u = 2^-24 ~ 6e-8):
  * draws of O(1) targets: every leapfrog step rounds each element about once (|x| <~ 5): ~3e-7 per step and
    draw, carried from draw to draw -> 2e-5 (L + 1) per draw taken, times the target's scale;
  * log densities: sums of D terms of size ~1 in fp32 (relative 1e-5) plus the energy error below -> 1e-5
    relative + 1e-3 sqrt(D) absolute;
  * tie margin tau of the accept test: a chain is compared until its first accept decision that differs from the
    oracle's, and such a flip must lie within tau of the oracle's threshold (|log u - Delta| < tau).  The position
    form recovers the momentum as eps rho_L = (c/2) x_L - x_{L-1}, which cancels: each element carries an error of
    about 2^-24 |x| / eps, the kinetic energy about D 2^-24 |x| rho / eps; with |x| rho <~ 16 that is
    tau = 1e-3 + 16 D 2^-24 / eps (1.6e-2 at D = 512, eps = 2^-5).  The velocity form, MALA and RW lose no digits
    that way: tau = 1e-3 + 4 D 2^-24.
At least 97 % of the chains must be compared through every draw, so no case passes by excluding everything.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _dev import np_
from oracle import philox as ph
from oracle import samplers as osm
from oracle.models import DiagGauss, GaussPriorLik, IsoGauss, Tempered

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- lane layouts of the fused separable samplers (sampler_sep.cu: launch_mk, sampler_sep_narrow.cu) -------------
ISO_D = {"1x1": [1, 4], "4x1": [5, 12, 13, 16], "8x1": [17, 28, 29, 32], "4x4": [33, 50, 60],
         "narrow": [61, 64, 76, 77, 92, 93, 100, 108], "8x4": [109, 124, 125, 128],
         "32x2": [129, 252, 253, 256], "32x4": [257, 508, 509, 512]}
DIAG_D = {"1x1": [3], "4x1": [13], "8x1": [30], "4x4": [33, 61, 64], "8x4": [65, 100, 125, 128], "32x2": [200],
          "32x4": [300]}
ALL_ISO = [d for v in ISO_D.values() for d in v]
ALL_DIAG = [d for v in DIAG_D.values() for d in v]
# one D per layout for the wider sweeps of algorithm parameters
ONE_ISO = [4, 13, 29, 50, 61, 77, 93, 125, 253, 509]


def sep_layout(D, iso, wide=True, narrow=True):
    """(G, J) of the fp32 fused sampler for dimension D (mirrors launch_mk / launch_sep_narrow)."""
    need = (D + 3) // 4 + 1
    if iso and narrow and 16 < need <= 28:
        return 4, {5: 5, 6: 6}.get((need + 3) // 4, 7)
    for lim, gj in ((4, (1, 1)), (16, (4, 1)), (32, (8, 1))):
        if D <= lim:
            return gj
    if wide and 64 < D <= 128:
        return 8, 4
    if wide and 32 < D <= 64:
        return 4, 4
    for lim, gj in ((64, (16, 1)), (128, (32, 1)), (256, (32, 2)), (512, (32, 4))):
        if D <= lim:
            return gj
    raise ValueError(D)


def ragged_chains(G):
    """Two CTAs' worth (at least 64 chains) plus three: the last CTA has lanes that shadow chain C - 1."""
    cpb = 128 // G
    return cpb * max(2, -(-64 // cpb)) + 3


def f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def tie_margin(D, eps=None):
    return 1e-3 + (16 * D * U / eps if eps is not None else 4 * D * U)


def dev_init_normal(bk, C, D, dtype, seed, chain_offset, draw):
    """bk_init_normal: [C, D] normals of (seed, global chain chain_offset + c, draw)."""
    from bayes_kit_b200 import _lib as L
    out = torch.empty(C, D, dtype=dtype, device="cuda")
    L.check(L.lib().bk_init_normal(out.data_ptr(), C, D, L.BK_F32 if dtype == torch.float32 else L.BK_F64,
                                   seed, chain_offset, draw, torch.cuda.current_stream().cuda_stream))
    return out


def philox_accept_uniforms(seed, chain_offset, n, C, D):
    """[n, C] accept uniforms of the single-uniform samplers in Philox mode (device_rng.cuh: accept_block)."""
    ch = np.uint64(chain_offset) + np.arange(C, dtype=np.uint64)
    return np.stack([ph.accept_uniform(seed, ch, t, D) for t in range(n)])


def check_vs_oracle(th0, d, l, a, od, ol, oa, ratio, us, draw_tol, tau, lp_atol):
    """Per-draw comparison with the tie rule of the module docstring.  Returns (max draw err, max logp err, kept)."""
    d, l, a = np_(d).astype(np.float64), np_(l).astype(np.float64), np_(a).astype(bool)
    prev = np.asarray(th0, dtype=np.float32)
    same = np.ones(a.shape[1], dtype=bool)
    logu = np.log(us)
    e_d = e_l = 0.0
    d32 = d.astype(np.float32)
    for t in range(a.shape[0]):
        flip = same & (a[t] != oa[t])
        bad = flip & (np.abs(logu[t] - ratio[t]) >= tau)
        assert not bad.any(), (f"draw {t}: accept decision differs away from a tie at chains {np.where(bad)[0][:8]}: "
                               f"log u - Delta = {(logu[t] - ratio[t])[bad][:4]}, tau = {tau:.3g}")
        same &= ~flip
        assert same.mean() >= 0.97, f"draw {t}: only {same.mean():.3f} of the chains still compared"
        # a rejected draw is the previous state, bit for bit
        rej = ~a[t]
        assert np.array_equal(d32[t][rej], prev[rej]), f"draw {t}: a rejected draw is not the previous state"
        prev = d32[t]
        err = np.abs(d[t][same] - od[t][same]).max(initial=0.0)
        assert err <= draw_tol * (t + 1), f"draw {t}: max |draw - oracle| = {err:.3g} > {draw_tol * (t + 1):.3g}"
        lerr = np.abs(l[t][same] - ol[t][same])
        assert (lerr <= 1e-5 * np.abs(ol[t][same]) + lp_atol).all(), f"draw {t}: max |logp - oracle| = {lerr.max():.3g}"
        e_d, e_l = max(e_d, err / (t + 1)), max(e_l, lerr.max(initial=0.0))
    return e_d, e_l, same.mean()


def run_sep(bk, algo, D, n, seed, *, iso=True, eps=0.2, L=10, sigma=1.0, metric=False, hastings=False):
    """One injected-stream run of a fused fp32 sampler and the fp64 oracle on the same (fp32-representable)
    values.  Returns (init, draws, logp, accept flags, oracle (draws, logp, accept, log ratio), uniforms)."""
    rng = np.random.default_rng(seed)
    G, _ = sep_layout(D, iso)
    C = ragged_chains(G)
    th0 = f32(rng.normal(size=(C, D)) * sigma)
    zs, us = f32(rng.standard_normal((n, C, D))), f32(rng.random((n, C)))
    if iso:
        om, dm = IsoGauss(D, sigma), bk.IsoGauss(D, sigma, dtype=torch.float32)
        om._prec = float(np.float32(om._prec))          # the device holds 1 / sigma^2 in fp32
    else:
        mu, prec = f32(rng.normal(size=D)), f32(rng.uniform(0.5, 2.0, D))
        om, dm = DiagGauss(mu, prec), bk.DiagGauss(mu, prec, dtype=torch.float32)
    m = f32(rng.uniform(0.5, 1.5, D)) if metric else None
    if algo == "hmc":
        s = bk.HMCDiag(dm, eps, L, metric_diag=m, init=th0)
        o = osm.hmc_diag_batch(om, th0, zs, us, float(np.float32(eps)), L, m, with_ratio=True)
    elif algo == "mala":
        s = bk.MALA(dm, eps, init=th0)
        o = osm.mala_batch(om, th0, zs, us, eps, with_ratio=True)
    else:
        prop = bk.GaussianRW(eps)
        s = bk.MetropolisHastings(dm, prop, prop.transition_lp, init=th0) if hastings else bk.Metropolis(dm, prop, init=th0)
        o = osm.metropolis_rw_batch(om, th0, zs, us, eps, hastings, with_ratio=True)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    return th0, d, l, s.last_accept, o, us


def _position_form(algo, iso, eps, L, metric, sigma=1.0):
    return algo == "hmc" and iso and not metric and L > 0 and np.float32(eps) ** 2 / sigma ** 2 >= 2.0 ** -10


def _check(bk, algo, D, *, iso=True, eps=0.2, L=10, sigma=1.0, metric=False, hastings=False, n=4):
    th0, d, l, a, (od, ol, oa, ratio), us = run_sep(bk, algo, D, n, 1000 * D + L + int(1e4 * eps), iso=iso, eps=eps,
                                                     L=L, sigma=sigma, metric=metric, hastings=hastings)
    pos = _position_form(algo, iso, eps, L, metric, sigma)
    tau = tie_margin(D, eps if pos else None)
    steps = L + 1 if algo == "hmc" else 1
    return check_vs_oracle(th0, d, l, a, od, ol, oa, ratio, us, 2e-5 * steps * max(1.0, sigma), tau,
                           1e-3 * np.sqrt(D) + (tau if pos else 0.0))


# ---- a. the stream itself ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [1, 3, 4, 6, 13, 50, 101])
def test_init_normal_stream(bk, D):
    """bk_init_normal against the restatement: element e is word e % 4 of block e // 4, fp64 exactly as
    philox_normal4<double>, fp32 as box_muller4 up to the approximate SFU instructions."""
    C = 37
    for seed, off, draw in ((0, 0, 0), (12345, 3, 7), (0xFFFFFFFF00000001, 1000, 0xFFFFFFFF)):
        got = np_(dev_init_normal(bk, C, D, torch.float64, seed, off, draw))
        want = ph.init_normal(seed, off, draw, C, D, np.float64)
        np.testing.assert_allclose(got, want, rtol=1e-13, atol=1e-14)
        got = np_(dev_init_normal(bk, C, D, torch.float32, seed, off, draw)).astype(np.float64)
        want = ph.init_normal(seed, off, draw, C, D, np.float32)
        err = np.abs(got - want)
        assert (err <= ph.box_muller4_tolerance(want)).all(), f"max fp32 normal error {err.max():.3g}"
        assert err.max() < 2e-4


# ---- b. fused separable samplers, fp32, injected streams vs the fp64 oracle ----------------------------------------
@pytest.mark.parametrize("D", ALL_ISO)
@pytest.mark.parametrize("algo", ["hmc", "mala", "rw"])
def test_sep_iso_vs_oracle(bk, algo, D):
    """HMC in the position form (eps = 0.2, L = 10), MALA and RW Metropolis on IsoGauss(D) in every layout."""
    eps = {"hmc": 0.2, "mala": 0.1, "rw": 2.4 / np.sqrt(D)}[algo]
    _check(bk, algo, D, eps=eps)


@pytest.mark.parametrize("D", ONE_ISO)
@pytest.mark.parametrize("eps,L", [(0.2, 1), (0.2, 2), (0.2, 3), (2.0 ** -5, 10), (2.0 ** -5, 3), (0.0312, 10),
                                   (0.2, 0)])
def test_sep_iso_hmc_forms(bk, D, eps, L):
    """Both parities of L in the position form, eps = 2^-5 (eps^2 prec = 2^-10 exactly: position form), 0.0312
    (velocity form), L = 0."""
    _check(bk, "hmc", D, eps=eps, L=L)


@pytest.mark.parametrize("D", ONE_ISO)
def test_sep_iso_sigma_and_mh(bk, D):
    """IsoGauss with sigma != 1 (prec = 1 / sigma^2 != 1) and MetropolisHastings with the symmetric transition lp."""
    _check(bk, "hmc", D, eps=0.3, L=5, sigma=1.5)
    _check(bk, "mala", D, eps=0.15, sigma=1.5)
    _check(bk, "rw", D, eps=2.0 / np.sqrt(D), hastings=True)


@pytest.mark.parametrize("D", ALL_DIAG)
def test_sep_diag_vs_oracle(bk, D):
    """DiagGauss: HMC with and without metric_diag, MALA."""
    _check(bk, "hmc", D, iso=False, eps=0.15, L=6)
    _check(bk, "hmc", D, iso=False, eps=0.15, L=5, metric=True)
    _check(bk, "mala", D, iso=False, eps=0.05)


# ---- c. Philox mode == injected reconstruction, bit for bit ------------------------------------------------------
def philox_vs_injected(bk, make, D, dtype, seed, chain_offset, n, n_uniform=None):
    """Run `make(init, seed, chain_offset)` in Philox mode and again fed the normals of bk_init_normal and the
    uniforms of the restatement; returns both results."""
    rng = np.random.default_rng(D)
    G, _ = sep_layout(D, True)
    C = ragged_chains(G)
    th0 = f32(rng.normal(size=(C, D)))
    s = make(th0, seed, chain_offset)
    d1, l1 = s.sample_n(n)
    a1 = s.last_accept
    zs = torch.stack([dev_init_normal(bk, C, D, dtype, seed, chain_offset, t) for t in range(n)])
    if n_uniform is None:
        us = philox_accept_uniforms(seed, chain_offset, n, C, D)
    else:
        ch = np.uint64(chain_offset) + np.arange(C, dtype=np.uint64)
        us = np.stack([np.stack([ph.philox_uniform(seed, k, ch, t) for k in range(n_uniform)], -1) for t in range(n)])
    s2 = make(th0, seed, chain_offset)
    d2, l2 = s2.sample_n(n, normals=zs, uniforms=us)
    return (np_(d1), np_(l1), np_(a1)), (np_(d2), np_(l2), np_(s2.last_accept)), s, s2


@pytest.mark.parametrize("D", ALL_ISO)
def test_philox_equals_injected_reconstruction(bk, D):
    """The in-kernel normals and accept uniform (spare-slot shuffle when ceil(D/4) < G J, philox_accept_uniform
    otherwise) are exactly bk_init_normal's normals and word 0 of block ceil(D/4): draws, logp, accept bitwise."""
    seed = 0x5EED0000 + D
    for algo in ("hmc", "mala", "rw"):
        def make(th0, sd, off):
            m = bk.IsoGauss(D, dtype=torch.float32)
            if algo == "hmc":
                return bk.HMCDiag(m, 0.2, 3, init=th0, seed=sd, chain_offset=off)
            if algo == "mala":
                return bk.MALA(m, 0.1, init=th0, seed=sd, chain_offset=off)
            return bk.Metropolis(m, bk.GaussianRW(2.4 / np.sqrt(D)), init=th0, seed=sd, chain_offset=off)
        for off in (0, 1 << 20):
            (d1, l1, a1), (d2, l2, a2), _, _ = philox_vs_injected(bk, make, D, torch.float32, seed, off, 3)
            assert np.array_equal(a1, a2), f"{algo} off={off}: accept flags differ"
            assert a1.any()
            assert np.array_equal(d1, d2), f"{algo} off={off}: draws differ"
            assert np.array_equal(l1, l2), f"{algo} off={off}: logp differs"


@pytest.mark.parametrize("D", ALL_DIAG)
def test_philox_equals_injected_diag(bk, D):
    rng = np.random.default_rng(D)
    mu, prec = f32(rng.normal(size=D)), f32(rng.uniform(0.5, 2.0, D))

    def make(th0, sd, off):
        return bk.HMCDiag(bk.DiagGauss(mu, prec, dtype=torch.float32), 0.15, 4, init=th0, seed=sd, chain_offset=off)
    (d1, l1, a1), (d2, l2, a2), _, _ = philox_vs_injected(bk, make, D, torch.float32, 77 + D, 5, 3)
    assert np.array_equal(a1, a2) and np.array_equal(d1, d2) and np.array_equal(l1, l2)


# ---- d. the diagnostic layout switches, in a child process ---------------------------------------------------------
def _child(tmp_path, env, fn, *args):
    """Run tests/test_gpu_fp32_parity.<fn>(*args, out) in a fresh interpreter with `env` added: the layout
    switches are read once per process into function-local statics."""
    out = str(tmp_path / f"{fn}.npz")
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
            f"import test_gpu_fp32_parity as t; t.{fn}(*{args!r}, out={out!r})\n")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    r = subprocess.run(cmd, env={**os.environ, **env}, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, f"child {env} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    return np.load(out)


def philox_runs(dims, out=None):
    """Philox-mode HMC (position form), MALA and RW on IsoGauss(D) for each D; returns / saves the results."""
    import bayes_kit_b200 as bk
    res = {}
    for D in dims:
        rng = np.random.default_rng(D)
        C = 67
        th0 = f32(rng.normal(size=(C, D)))
        m = bk.IsoGauss(D, dtype=torch.float32)
        for algo, s in (("hmc", bk.HMCDiag(m, 0.2, 5, init=th0, seed=D, chain_offset=3)),
                        ("mala", bk.MALA(m, 0.1, init=th0, seed=D, chain_offset=3)),
                        ("rw", bk.Metropolis(m, bk.GaussianRW(2.4 / np.sqrt(D)), init=th0, seed=D, chain_offset=3))):
            d, l = s.sample_n(4)
            res[f"{algo}_{D}_d"], res[f"{algo}_{D}_l"], res[f"{algo}_{D}_a"] = np_(d), np_(l), np_(s.last_accept)
    if out:
        np.savez(out, **res)
    return res


def _same_until_decisions_differ(ref, got, key):
    """Accept decisions equal away from ties (>= 97 % of the chains agree throughout) and the draws bitwise equal
    while a chain's decision history agrees: the elementwise arithmetic does not depend on the layout, only the
    group reductions (and with them the last bits of Delta and logp) do."""
    a0, a1 = ref[key + "_a"].astype(bool), got[key + "_a"].astype(bool)
    agree = np.logical_and.accumulate(a0 == a1, axis=0)
    assert agree[-1].mean() >= 0.97, f"{key}: decisions differ in {1 - agree[-1].mean():.3f} of the chains"
    for t in range(a0.shape[0]):
        assert np.array_equal(ref[key + "_d"][t][agree[t]], got[key + "_d"][t][agree[t]]), f"{key}: draw {t} differs"
        np.testing.assert_allclose(got[key + "_l"][t][agree[t]], ref[key + "_l"][t][agree[t]], rtol=2e-6, atol=1e-4)


@pytest.mark.parametrize("env,dims", [({"BK_SEP_LAYOUT": "0"}, [61, 64, 77, 93, 100, 108]),
                                      ({"BK_SEP_WIDE": "0"}, [33, 50, 64, 65, 100, 128])])
def test_sep_layout_switches(bk, tmp_path, env, dims):
    """BK_SEP_LAYOUT=0 (power-of-two layouts instead of 4x5..4x7) and BK_SEP_WIDE=0 (16x1 / 32x1 instead of 4x4 /
    8x4) run the same chains as the default layouts."""
    ref = philox_runs(dims)
    got = _child(tmp_path, env, "philox_runs", dims)
    for D in dims:
        for algo in ("hmc", "mala", "rw"):
            _same_until_decisions_differ(ref, got, f"{algo}_{D}")


# ---- e. fused DrGHMC, fp32 -------------------------------------------------------------------------------------
DR_D = [3, 13, 30, 40, 64, 65, 128, 200]


@pytest.mark.parametrize("D", DR_D)
@pytest.mark.parametrize("K,retry", [(2, True), (3, False), (3, True)])
def test_drghmc_vs_oracle(bk, D, K, retry):
    """The fused DrGHMC kernel in fp32 (layouts 1x1 .. 32x2, the fp32-only 4x4 and 8x4) against osm.drghmc under
    injected streams.  Nested accept / retry tests have no single Delta: a chain is compared until its first
    differing decision (accept flag or uniforms consumed), and 97 % of the chains must be compared throughout."""
    rng = np.random.default_rng(D * 10 + K)
    G, _ = sep_layout(D, False)
    C, n = ragged_chains(G), 3
    iso = D % 2 == 1
    if iso:
        om, dm = IsoGauss(D), bk.IsoGauss(D, dtype=torch.float32)
    else:
        mu, prec = f32(rng.normal(size=D)), f32(rng.uniform(0.5, 2.0, D))
        om, dm = DiagGauss(mu, prec), bk.DiagGauss(mu, prec, dtype=torch.float32)
    eps0 = 1.6 * D ** -0.25                  # a first proposal that is often rejected: retries happen
    sizes, counts = [float(np.float32(eps0 / 2 ** k)) for k in range(K)], [4 * 2 ** k for k in range(K)]
    damp = float(np.float32(0.2))
    th0, rho0 = f32(rng.normal(size=(C, D))), f32(rng.normal(size=(C, D)))
    zs, us = f32(rng.standard_normal((n, C, D))), f32(rng.random((n, C, 2 * K)))
    od, ol, orho, oused = osm.drghmc_batch(om, th0, rho0, zs, us, K, sizes, counts, damp, None, retry)
    s = bk.DrGhmcDiag(dm, K, sizes, counts, damp, init=th0, prob_retry=retry)
    s.set_momentum(rho0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    d, l, a, used = np_(d).astype(np.float64), np_(l).astype(np.float64), np_(s.last_accept), np_(s.last_n_uniform)
    # oracle accept flags: the draw moved
    prev, oa = th0, np.zeros((n, C), dtype=bool)
    for t in range(n):
        oa[t] = np.any(od[t] != prev, axis=1)
        prev = od[t]
    same = np.ones(C, dtype=bool)
    for t in range(n):
        same &= (a[t].astype(bool) == oa[t]) & (used[t] == oused[t])
        assert same.mean() >= 0.97, f"draw {t}: decisions differ in {1 - same.mean():.3f} of the chains"
        tol = 2e-5 * (sum(counts) + 1) * (t + 1)
        assert np.abs(d[t][same] - od[t][same]).max() <= tol
        np.testing.assert_allclose(l[t][same], ol[t][same], rtol=1e-5, atol=1e-3 * np.sqrt(D))
    assert (oused > 2).any()                  # the case exercises a second proposal
    np.testing.assert_allclose(np_(s.rho)[same].astype(np.float64), orho[same], atol=2e-5 * (sum(counts) + 1) * n)


@pytest.mark.parametrize("D", DR_D)
def test_drghmc_philox_equals_injected(bk, D):
    """DrGHMC in Philox mode == fed bk_init_normal's normals and philox_uniform(k) of TAG_UNIFORM, bitwise."""
    K = 3
    iso = D % 2 == 1
    rng = np.random.default_rng(D)
    mu, prec = f32(rng.normal(size=D)), f32(rng.uniform(0.5, 2.0, D))

    def make(th0, sd, off):
        m = bk.IsoGauss(D, dtype=torch.float32) if iso else bk.DiagGauss(mu, prec, dtype=torch.float32)
        return bk.DrGhmcDiag(m, K, [0.3, 0.15, 0.075], [4, 8, 16], 0.2, init=th0, seed=sd, chain_offset=off)
    (d1, l1, a1), (d2, l2, a2), s1, s2 = philox_vs_injected(bk, make, D, torch.float32, 99 + D, 11, 3, n_uniform=2 * K)
    assert np.array_equal(np_(s1.last_n_uniform), np_(s2.last_n_uniform))
    assert np.array_equal(a1, a2) and np.array_equal(d1, d2) and np.array_equal(l1, l2)
    assert np.array_equal(np_(s1.rho), np_(s2.rho))


# ---- f. SMC move kernel, fp32, per temperature vs the oracle --------------------------------------------------------
SMC_CASES = [(3, "rw"), (12, "rw"), (30, "rw"), (45, "rw"), (50, "rw"), (52, "rw"), (64, "rw"), (100, "rw"),
             (200, "rw"), (5, "mala"), (45, "mala"), (100, "mala"), (12, "hmc"), (50, "hmc"), (130, "hmc")]
CDF_MARGIN = 1e-5     # fraction of the total weight: closer resample thresholds may go either way in fp32


def _oracle_move(om, th, t0, z, kernel):
    """Proposal and log acceptance ratio of one SMC move at temperature t0 (oracle.samplers.smc_move)."""
    tm = Tempered(om, t0)
    if kernel[0] == "rw":
        star = th + kernel[1] * z
        return star, tm.log_density(star) - tm.log_density(th)
    tiny = np.array([1e-300])         # log u = -690: the proposal is taken unless Delta is not a number
    if kernel[0] == "mala":
        d, _, _, r = osm.mala(tm, th, z[None], tiny, kernel[1], with_ratio=True)
    else:
        d, _, _, r = osm.hmc_diag(tm, th, z[None], tiny, kernel[1], kernel[2], with_ratio=True)
    return d[0], r[0]


def smc_check(D, kind, resample, T=4, out=None):
    """Runs T temperatures of the fp32 SMC under injected streams; before each, the oracle restarts from the
    device's own particles (so that rounding does not compound).  Asserts, per temperature: the accept flags
    (flips only within the tie margin), the resample indices (except thresholds within CDF_MARGIN of a CDF edge)
    and the particles.  Returns the worst errors seen."""
    import bayes_kit_b200 as bk
    rng = np.random.default_rng(D * 7 + len(kind) + len(resample))
    M = 300
    m0, p0 = f32(rng.normal(size=D) * 0.1), f32(rng.uniform(0.5, 1.5, D))
    mu, pl = f32(rng.normal(size=D)), f32(rng.uniform(1.0, 4.0, D) / np.sqrt(D / 4 + 1))
    om = GaussPriorLik(m0, p0, mu, pl)
    dm = bk.GaussPriorLik(m0, p0, mu, pl, dtype=torch.float32)
    scale = float(np.float32({"rw": 1.5, "mala": 0.3, "hmc": 0.3}[kind] / np.sqrt(D)))
    kernel = {"rw": ("rw", scale), "mala": ("mala", scale), "hmc": ("hmc", scale, 3)}[kind]
    bkern = {"rw": lambda: bk.metropolis_kernel(scale), "mala": lambda: bk.mala_kernel(scale),
             "hmc": lambda: bk.hmc_kernel(scale, 3)}[kind]()
    th0 = f32(rng.normal(size=(M, D)))
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, bkern, resample=resample)
    tau = tie_margin(D)
    worst = {"theta": 0.0, "skipped_idx": 0, "ties": 0, "min_margin": np.inf}
    for n in range(1, T + 1):
        t0 = float(np.float32((n - 1) / T))
        cur = np_(smc.thetas).astype(np.float64)
        zs, au, ru = f32(rng.standard_normal((M, D))), f32(rng.random(M)), f32(rng.random(M))
        prop, ratio = zip(*[_oracle_move(om, cur[m], t0, zs[m], kernel) for m in range(M)])
        prop, ratio = np.stack(prop), np.array(ratio)
        oa = np.log(au) < ratio
        smc.transition(n, normals=zs, acc_uniforms=au, res_uniforms=ru if resample == "multinomial" else ru[:1])
        a = np_(smc.last_accept).astype(bool)
        flip = a != oa
        tie = np.abs(np.log(au) - ratio) < tau
        assert not (flip & ~tie).any(), f"n={n}: accept flags differ away from a tie at {np.where(flip & ~tie)[0][:8]}"
        worst["ties"] += int(flip.sum())
        moved = np.where(a[:, None], prop, cur)             # the device's decisions: no cascade from a tie
        idx = np_(smc.last_indices).astype(np.int64)
        if resample == "multinomial":
            w = osm.smc_weights(om, moved, n, T)
            want, cdf = osm.multinomial_indices(w, ru)
            lo = np.where(want > 0, cdf[np.maximum(want - 1, 0)], 0.0)
            margin = np.minimum(np.abs(ru - lo), np.abs(cdf[np.minimum(want, M - 1)] - ru))
        else:
            t1 = n / T
            logw = np.array([(om.log_likelihood(th) * t1 + om.log_prior(th)) -
                             (om.log_likelihood(th) * t0 + om.log_prior(th)) for th in moved])
            want, cum = osm.systematic_indices(logw, ru[0])
            W = float(cum[-1])
            thr = np.minimum(np.floor((np.arange(M) + ru[0]) * (W / M)), W - 1)
            lo = np.where(want > 0, cum[np.maximum(want - 1, 0)], 0.0)
            margin = np.minimum(np.abs(thr - lo), np.abs(cum[want] - thr)) / W
        near = margin < CDF_MARGIN
        worst["min_margin"] = min(worst["min_margin"], float(margin.min()))
        worst["skipped_idx"] += int(near.sum())
        assert np.array_equal(idx[~near], want[~near]), f"n={n}: resample indices differ at {np.where((idx != want) & ~near)[0][:8]}"
        # a threshold lands within CDF_MARGIN of one of the M edges with probability ~2 M CDF_MARGIN (0.6 %)
        assert near.mean() < 0.05, f"n={n}: {near.sum()} resample thresholds within the margin"
        got = np_(smc.thetas).astype(np.float64)
        steps = kernel[2] + 1 if kind == "hmc" else 1
        err = np.abs(got - moved[idx]).max()
        worst["theta"] = max(worst["theta"], float(err))
        assert err <= 2e-5 * steps * max(1.0, np.abs(moved).max() / 3), f"n={n}: particles differ by {err:.3g}"
    if out:
        np.savez(out, **{k: np.float64(v) for k, v in worst.items()})
    return worst


@pytest.mark.parametrize("D,kind", SMC_CASES)
@pytest.mark.parametrize("resample", ["systematic", "multinomial"])
def test_smc_move_vs_oracle(bk, D, kind, resample):
    smc_check(D, kind, resample)


@pytest.mark.parametrize("env", [{"BK_SMC_LAYOUT": "0"}, {"BK_SMC_LAYOUT": "1"}, {"BK_SMC_OCC": "2"},
                                 {"BK_SMC_OCC": "4"}, {"BK_SEP_WIDE": "0"}])
def test_smc_layout_switches_vs_oracle(bk, tmp_path, env):
    """The diagnostic SMC layouts (16x4 / 8x2 lanes, the occupancy-capped 4x4 variants, no wide layout) against
    the oracle, each in its own process."""
    for D in (45, 50, 52, 64):
        _child(tmp_path, env, "smc_check", D, "rw", "systematic")
