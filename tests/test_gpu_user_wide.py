"""User models from 33 to USER_WIDE_MAX_D dims: the wide HMCDiag / MALA / RW-Metropolis kernels (trajectory in shared
memory, state in the generic engine's cache).  Parity runs fp64 with injected streams against the NumPy oracle, and
against the generic engine (BK_FORCE_GENERIC=1) and the built-in DiagGauss plugin on the same Philox words."""
import ctypes as C

import numpy as np
import pytest
import torch

from _dev import np_
from _user_cuda import (BANANA, DIAG, FUSED_MAX_D, PRIOR_LIK_WEIGHTED, WIDE_MAX_D, NpPriorLik, banana, check,
                        diag_params, run_split, same, streams_uniforms_last)
from oracle import samplers as osm
from oracle.models import DiagGauss as ODiag

pytestmark = pytest.mark.gpu

DIMS = sorted({33, 64, WIDE_MAX_D})


@pytest.fixture(autouse=True)
def _wide_engine(monkeypatch):
    monkeypatch.setenv("BK_FORCE_GENERIC", "0")


# ---- 1. against the oracle, fp64, injected streams ------------------------------------------------------------------
@pytest.mark.parametrize("C_", [1, 37, 100])
@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("L", [0, 1, 7])
@pytest.mark.parametrize("metric", [False, True])
def test_hmc_matches_oracle(bk, C_, D, L, metric):
    n = 4
    dm, om = banana(bk, D, dot=True)
    th0, zs, us = streams_uniforms_last(C_, D, n, D + L)
    m = np.random.default_rng(D).uniform(0.5, 2.0, D) if metric else None
    eps = 0.6 / D ** 0.25
    s = bk.HMCDiag(dm, eps, L, metric_diag=m, init=th0)
    assert "bk_user_wide_hmc" in s.compile_log
    d, l, a = run_split(s, zs, us, 2)
    check(d, l, a, osm.hmc_diag_batch(om, th0, zs, us, eps, L, m))
    np.testing.assert_allclose(np_(s.theta), np_(d[-1]).reshape(np_(s.theta).shape), rtol=0, atol=0)


@pytest.mark.parametrize("C_", [1, 37, 100])
@pytest.mark.parametrize("D", DIMS)
def test_mala_matches_oracle(bk, C_, D):
    n = 6
    dm, om = banana(bk, D, dot=True)
    th0, zs, us = streams_uniforms_last(C_, D, n, 11 + D)
    eps = 0.4 / D ** (1 / 3)
    s = bk.MALA(dm, eps, init=th0)
    assert "bk_user_wide_mala" in s.compile_log
    d, l, a = run_split(s, zs, us, 3)
    check(d, l, a, osm.mala_batch(om, th0, zs, us, eps))


@pytest.mark.parametrize("C_", [1, 37, 100])
@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("hastings", [False, True])
def test_metropolis_matches_oracle(bk, C_, D, hastings):
    n = 6
    dm, om = banana(bk, D, dot=True)
    th0, zs, us = streams_uniforms_last(C_, D, n, 12 + D)
    scale = 1.5 / D ** 0.5
    prop = bk.GaussianRW(scale)
    s = bk.MetropolisHastings(dm, prop, prop.transition_lp, init=th0) if hastings else bk.Metropolis(dm, prop, init=th0)
    assert "bk_user_wide_mh" in s.compile_log
    d, l, a = run_split(s, zs, us, 3)
    check(d, l, a, osm.metropolis_rw_batch(om, th0, zs, us, scale, hastings))


def test_prior_lik_matches_oracle(bk):
    C_, D, n = 37, 40, 5
    w = np.random.default_rng(4).uniform(0.5, 2.0, D)
    dm = bk.CudaPriorLikModel(PRIOR_LIK_WEIGHTED, D, params=w, dtype=torch.float64)
    om = NpPriorLik(w)
    th0, zs, us = streams_uniforms_last(C_, D, n, 31)
    s = bk.HMCDiag(dm, 0.15, 5, init=th0)
    assert "bk_user_wide_hmc" in s.compile_log
    d, l, a = run_split(s, zs, us, 2)
    check(d, l, a, osm.hmc_diag_batch(om, th0, zs, us, 0.15, 5))
    s = bk.MALA(dm, 0.05, init=th0)
    d, l, a = run_split(s, zs, us, 2)
    check(d, l, a, osm.mala_batch(om, th0, zs, us, 0.05))


# ---- 2. against the generic engine and the built-in plugin, Philox ---------------------------------------------------
def _samplers(bk, D):
    return (lambda m, init: bk.HMCDiag(m, 0.6 / D ** 0.25, 5, init=init, seed=17),
            lambda m, init: bk.MALA(m, 0.4 / D ** (1 / 3), init=init, seed=17),
            lambda m, init: bk.Metropolis(m, bk.GaussianRW(1.5 / D ** 0.5), init=init, seed=17),
            lambda m, init: bk.MetropolisHastings(m, *(lambda p: (p, p.transition_lp))(bk.GaussianRW(1.5 / D ** 0.5)),
                                                  init=init, seed=17))


@pytest.mark.parametrize("D", [64, WIDE_MAX_D])
def test_wide_equals_generic(bk, monkeypatch, D):
    dm, _ = banana(bk, D)
    init = np.random.default_rng(2).normal(size=(100, D))
    for make in _samplers(bk, D):
        monkeypatch.setenv("BK_FORCE_GENERIC", "0")
        a = make(dm, init)
        da, la = a.sample_n(10)
        monkeypatch.setenv("BK_FORCE_GENERIC", "1")
        b = make(dm, init)
        db, lb = b.sample_n(10)
        same(a, b, da, db, la, lb)


def test_switching_engines_keeps_the_chains(bk, monkeypatch):
    """wide -> generic -> wide call by call on one sampler gives the generic engine's chains: the wide kernels keep the
    generic engine's (lp, grad) cache valid, and read it back."""
    D = 48
    dm, _ = banana(bk, D)
    init = np.random.default_rng(6).normal(size=(70, D))
    for make in _samplers(bk, D):
        monkeypatch.setenv("BK_FORCE_GENERIC", "1")
        ref = make(dm, init)
        want = [ref.sample_n(4) + (ref.last_accept.clone(),) for _ in range(3)]
        s = make(dm, init)
        for k, eng in enumerate(("0", "1", "0")):
            monkeypatch.setenv("BK_FORCE_GENERIC", eng)
            d, l = s.sample_n(4)
            assert torch.equal(s.last_accept, want[k][2])
            np.testing.assert_allclose(np_(d), np_(want[k][0]), rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(np_(l), np_(want[k][1]), rtol=1e-12, atol=1e-12)


def test_user_diag_gauss_equals_builtin(bk):
    D = 64
    mu, pr = diag_params(D)
    user = bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]), dtype=torch.float64)
    built = bk.DiagGauss(mu, pr, dtype=torch.float64)
    init = np.random.default_rng(D).normal(size=(64, D))
    for make in _samplers(bk, D)[:3]:
        a, b = make(user, init), make(built, init)
        da, la = a.sample_n(20)
        db, lb = b.sample_n(20)
        same(a, b, da, db, la, lb)


def test_shard_invariant(bk):
    """chains 40 .. 99 on their own (chain_offset = 40, a different split into warps) are those of the full run"""
    D = 96
    dm, _ = banana(bk, D, dtype=torch.float32)
    init = np.random.default_rng(2).normal(size=(100, D))
    for make in (lambda init, **kw: bk.HMCDiag(dm, 0.2, 5, init=init, seed=9, **kw),
                 lambda init, **kw: bk.MALA(dm, 0.05, init=init, seed=9, **kw),
                 lambda init, **kw: bk.Metropolis(dm, bk.GaussianRW(0.15), init=init, seed=9, **kw)):
        full = make(init).sample_n(10)
        part = make(init[40:], chain_offset=40).sample_n(10)
        assert torch.equal(full[0][:, 40:], part[0])
        assert torch.equal(full[1][:, 40:], part[1])


# ---- 3. statistics, fp32 -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [64, 128])
def test_banana_moments(bk, D):
    """x1 has mean b and variance 1 + 2 b^2, every other coordinate is N(0, 1)"""
    b = 0.5
    dm = bk.CudaModel(BANANA, D, params=[b])
    s = bk.HMCDiag(dm, 0.25, 8, chains=2048, seed=3)
    s.sample_n(100, keep_draws=False)
    d, _ = s.sample_n(200)
    x = d.double()
    mean_t = torch.zeros(D, dtype=torch.float64, device=x.device)
    var_t = torch.ones(D, dtype=torch.float64, device=x.device)
    mean_t[1], var_t[1] = b, 1 + 2 * b * b
    for stat, want in ((x, mean_t), ((x - mean_t) ** 2, var_t)):
        ess = bk.ess(stat, draws_first=True).reshape(-1, D).sum(0)
        est = stat.mean((0, 1))
        mcse = stat.reshape(-1, D).std(0) / ess.sqrt()
        z = ((est - want) / mcse).abs()
        assert float(z.max()) < 4, (np_(est), np_(mcse))


# ---- 4. host paths and dispatch --------------------------------------------------------------------------------------
def test_host_draws_and_moments(bk):
    D = 80
    dm = bk.CudaModel(BANANA, D, params=[0.5])
    for make in (lambda: bk.HMCDiag(dm, 0.2, 4, chains=300, seed=4), lambda: bk.MALA(dm, 0.05, chains=300, seed=4),
                 lambda: bk.Metropolis(dm, bk.GaussianRW(0.15), chains=300, seed=4)):
        s = make()
        d1, _ = s.sample_n(9, moments=True)
        d2, _ = s.sample_n(7, moments=True)
        np.testing.assert_allclose(np_(s.running_rhat()), np_(bk.rhat(torch.cat([d1, d2]), draws_first=True)),
                                   rtol=1e-4)
        a, b = make(), make()
        da, la = a.sample_n(5)
        hd, hl = b.sample_host_n(5, chunk_chains=100)
        assert torch.equal(da.cpu(), hd) and torch.equal(la.cpu(), hl)


def test_compile_log_and_dispatch(bk, monkeypatch):
    lib = bk._lib.lib()
    for D, wide in ((FUSED_MAX_D, False), (FUSED_MAX_D + 1, True), (WIDE_MAX_D, True), (WIDE_MAX_D + 1, False)):
        dm, _ = banana(bk, D, dtype=torch.float32)
        log = C.create_string_buffer(b"stale", 1 << 20)
        assert lib.bk_user_wide_prepare(dm.handle, log, len(log)) == bk._lib.BK_OK
        assert ("bk_user_wide_hmc" in log.value.decode()) == wide
        for s in (bk.HMCDiag(dm, 0.1, 3, chains=8, seed=1), bk.MALA(dm, 0.05, chains=8, seed=1),
                  bk.Metropolis(dm, bk.GaussianRW(0.1), chains=8, seed=1)):
            if wide:
                assert all(k in s.compile_log for k in ("bk_user_wide_hmc", "bk_user_wide_mala", "bk_user_wide_mh"))
            else:
                assert s.compile_log == ""
            s.sample_n(2)
        # the generic engine needs scratch, the fused engines none
        assert (lib.bk_hmc_diag_workspace_bytes(dm.handle, 64) == 0) == (D <= WIDE_MAX_D)
    monkeypatch.setenv("BK_FORCE_GENERIC", "1")
    dm, _ = banana(bk, 64, dtype=torch.float32)
    assert bk.HMCDiag(dm, 0.1, 3, chains=8, seed=1).compile_log == ""
