"""CudaProposal(gradient=True): user-written CUDA proposals that read the model's gradient.  Engines: the fused
bk_user_mhp_grad (a user model with dims <= 32, compiled together with the proposal) and, for every other model, four
launches per draw (bk_user_propose_grad, the model's log density and gradient, bk_user_dh_grad, the accept test).
Proposals: MALA restated (against bk.MALA) and the Barker proposal (against the NumPy oracle)."""
import re

import numpy as np
import pytest
import torch

from _dev import np_
from _user_cuda import BANANA, BARKER, MALA_G, PRIOR_LIK, NpBanana
from bayes_kit_b200 import _lib as L
from oracle import models as om
from oracle import proposals as opr

pytestmark = pytest.mark.gpu


def np_barker(model, sigma):
    """The Barker proposal as a reference user writes it: closures over the model's gradient."""
    def softplus(x):
        return x + np.log1p(np.exp(-x)) if x > 0 else np.log1p(np.exp(x))

    def propose(th, z, u):
        g = model.log_density_gradient(th)[1]
        w = sigma * z
        keep = 1 / (1 + np.exp(-w * g))
        return th + np.where(u[:th.shape[0]] < keep, w, -w)

    def tld(to, frm):
        g = model.log_density_gradient(frm)[1]
        s = 0.0
        for e in range(to.shape[0]):
            w = to[e] - frm[e]
            r = w / sigma
            s -= 0.5 * r * r + softplus(-w * g[e])
        return s
    return propose, tld


def _mala_params(eps):
    return [eps, np.sqrt(2 * eps), -0.25 / eps]


def _banana(bk, D, dtype=torch.float64):
    return bk.CudaModel(BANANA, D, params=[0.5], dtype=dtype)


def _barker(bk, D, sigma, dtype=torch.float64):
    return bk.CudaProposal(BARKER, D, params=[sigma], uniforms=D, dtype=dtype, gradient=True)


def _launches():
    return int(L.lib().bk_launch_count())


def _close(a, b, tol):
    host = lambda x: x if isinstance(x, np.ndarray) else np_(x)   # noqa: E731
    np.testing.assert_allclose(host(a), host(b), rtol=tol, atol=tol)


# ---- 1. MALA restated as a gradient proposal equals bk.MALA ----------------------------------------------------------
@pytest.mark.parametrize("injected", [False, True])
@pytest.mark.parametrize("case", ["fused8", "fused32", "generic40", "forced8", "diag12"])
def test_mala_restated_equals_mala(bk, monkeypatch, case, injected):
    D = int(re.sub(r"\D", "", case))
    if case.startswith("forced"):
        monkeypatch.setenv("BK_FORCE_GENERIC", "1")
    if case.startswith("diag"):
        rng = np.random.default_rng(D)
        model = bk.DiagGauss(rng.normal(size=D), rng.uniform(0.5, 3.0, D), dtype=torch.float64)
    else:
        model = _banana(bk, D)
    eps, C_, n = 0.6 / D ** (1 / 3), 70, 8
    init = np.random.default_rng(D + 1).normal(size=(C_, D))
    prop = bk.CudaProposal(MALA_G, D, params=_mala_params(eps), dtype=torch.float64, gradient=True)
    a = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init, seed=9)
    b = bk.MALA(model, eps, init=init, seed=9)
    kw = {}
    if injected:
        rng = np.random.default_rng(7)
        kw = dict(normals=rng.standard_normal((n, C_, D)), uniforms=rng.random((n, C_, 1)))
    for _ in range(2):   # the second call starts from each engine's cached state
        da, la = a.sample_n(n, **kw)
        db, lb = b.sample_n(n, **kw)
        assert torch.equal(a.last_accept, b.last_accept)
        assert 0 < float(a.last_accept.float().mean()) < 1
        _close(da, db, 1e-12)
        _close(la, lb, 1e-12)


# ---- 2. oracle parity: the Barker proposal, fp64, injected streams ----------------------------------------------------
@pytest.mark.parametrize("D,C_,kind", [(1, 37, "diag"), (5, 1, "banana"), (5, 100, "diag"), (32, 100, "banana"),
                                       (40, 37, "banana")])
def test_barker_matches_oracle(bk, D, C_, kind):
    n, sigma = 6, 1.2 / np.sqrt(D)
    if kind == "banana":
        dev, npm = _banana(bk, D), NpBanana(D, 0.5)
    else:
        rng = np.random.default_rng(D)
        mu, pr = rng.normal(size=D), rng.uniform(0.5, 3.0, D)
        dev, npm = bk.DiagGauss(mu, pr, dtype=torch.float64), om.DiagGauss(mu, pr)
    prop = _barker(bk, D, sigma)
    rng = np.random.default_rng(D * 1000 + C_)
    th0 = rng.normal(size=(C_, D))
    zs, us = rng.standard_normal((n, C_, D)), rng.random((n, C_, 1 + D))
    propose, tld = np_barker(npm, sigma)
    s = bk.MetropolisHastings(dev, prop, prop.transition_lp, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    wd, wl, wa = opr.metropolis_hastings_batch(npm, th0, zs, us, propose, tld)
    assert np.array_equal(np_(s.last_accept).astype(bool), wa)
    assert 0 < wa.mean() < 1 or C_ == 1
    _close(d, wd, 1e-10)
    _close(l, wl, 1e-10)
    # Metropolis leaves out the Hastings term, as the reference's does for any proposal
    s = bk.Metropolis(dev, prop, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    wd, wl, wa = opr.metropolis_hastings_batch(npm, th0, zs, us, propose)
    assert np.array_equal(np_(s.last_accept).astype(bool), wa)
    _close(d, wd, 1e-10)


# ---- 3. the fused and the generic engine agree ------------------------------------------------------------------------
def test_fused_and_generic_agree(bk, monkeypatch):
    D, C_, n = 8, 200, 6
    model, prop = _banana(bk, D), _barker(bk, D, 0.6)
    init = np.random.default_rng(2).normal(size=(C_, D))
    make = lambda: bk.MetropolisHastings(model, prop, prop.transition_lp, init=init, seed=13)   # noqa: E731
    fused, generic, alt = make(), make(), make()
    assert "bk_user_mhp_grad" in fused.compile_log
    df, lf = fused.sample_n(2 * n)
    af = fused.last_accept
    monkeypatch.setenv("BK_FORCE_GENERIC", "1")
    dg, lg = generic.sample_n(2 * n)
    assert torch.equal(af, generic.last_accept)
    _close(df, dg, 1e-12)
    _close(lf, lg, 1e-12)
    # alternate the engines call by call: the chains carry on
    parts = []
    for k in range(4):
        monkeypatch.setenv("BK_FORCE_GENERIC", "1" if k % 2 else "0")
        parts.append(alt.sample_n(n // 2)[0])
    _close(torch.cat(parts), df, 1e-12)


# ---- 4. shards and the host surface -----------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [6, 40])
def test_shards_equal_one_sampler(bk, D):
    model, prop = _banana(bk, D, torch.float32), _barker(bk, D, 0.8 / np.sqrt(D), torch.float32)
    init = np.random.default_rng(D).normal(size=(96, D))
    full = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init, seed=4).sample_n(10)[0]
    lo = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init[:40], seed=4).sample_n(10)[0]
    hi = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init[40:], seed=4, chain_offset=40).sample_n(10)[0]
    assert torch.equal(full, torch.cat([lo, hi], 1))


@pytest.mark.parametrize("kind", ["user8", "user40", "diag"])
def test_host_draws_and_moments(bk, kind):
    if kind == "diag":
        rng = np.random.default_rng(12)
        model = bk.DiagGauss(rng.normal(size=12), rng.uniform(0.5, 3.0, 12))
    else:
        model = _banana(bk, int(kind[4:]), torch.float32)
    D = model.dims()
    prop = bk.CudaProposal(MALA_G, D, params=_mala_params(0.3), gradient=True)
    make = lambda: bk.MetropolisHastings(model, prop, prop.transition_lp, chains=300, seed=8)   # noqa: E731
    a, b, c = make(), make(), make()
    da, la = a.sample_n(5)
    db, lb = a.sample_n(3)
    hd, hl = b.sample_host_n(5, chunk_chains=128)   # the first draw in chain chunks
    hd2, hl2 = b.sample_host_n(3, chunk_chains=[100, 200])
    assert torch.equal(da.cpu(), hd) and torch.equal(la.cpu(), hl)
    assert torch.equal(db.cpu(), hd2) and torch.equal(lb.cpu(), hl2)
    h1, l1 = c.sample_host(chunk_chains=64)
    assert torch.equal(da[0].cpu(), h1) and torch.equal(la[0].cpu(), l1)
    s = make()
    d1, _ = s.sample_n(9, moments=True)
    d2, _ = s.sample_n(7, moments=True)
    mean, var, n = s.running_moments()
    x = torch.cat([d1, d2]).double()
    assert n == 16
    np.testing.assert_allclose(np_(mean), np_(x.mean(0)), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(np_(var), np_(x.var(0)), rtol=1e-7, atol=1e-9)
    np.testing.assert_allclose(np_(s.running_rhat()), np_(bk.rhat(x.permute(1, 0, 2))), rtol=1e-6, atol=1e-9)


# ---- 5. statistics, fp32 Philox ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [8, 40])
def test_barker_samples_the_banana(bk, D):
    """x0 ~ N(0, 1), x1 | x0 ~ N(b x0^2, 1) with b = 0.5, the rest N(0, 1): E x1 = b, Var x1 = 1 + 2 b^2."""
    model, prop = _banana(bk, D, torch.float32), _barker(bk, D, 1.6 / D ** (1 / 6), torch.float32)
    s = bk.MetropolisHastings(model, prop, prop.transition_lp, chains=4096, seed=17)
    s.sample_n(300, keep_draws=False)
    x = s.sample_n(300)[0].double()
    assert 0.1 < float(s.last_accept.float().mean()) < 0.98
    mean_t = torch.zeros(D, dtype=torch.float64, device="cuda")
    mean_t[1] = 0.5
    var_t = torch.ones(D, dtype=torch.float64, device="cuda")
    var_t[1] = 1.5
    for stat, want in ((x, mean_t), ((x - mean_t) ** 2, var_t)):
        ess = bk.ess(stat, draws_first=True).reshape(-1, D).sum(0)
        est = stat.mean((0, 1))
        z = ((est - want) / (stat.reshape(-1, D).std(0) / ess.sqrt())).abs()
        assert float(z.max()) < 4, (np_(est), np_(z))


# ---- 6. surface -------------------------------------------------------------------------------------------------------
def test_launch_counts_show_the_engine(bk):
    """fused: one launch per call; otherwise four per draw (three without the Hastings term) plus the evaluation of
    the (log p, grad log p) cache on the first call only."""
    for D, hastings, first, later in ((8, True, lambda n: 1, lambda n: 1), (40, True, lambda n: 4 * n + 1, lambda n: 4 * n),
                                      (40, False, lambda n: 3 * n + 1, lambda n: 3 * n)):
        model = _banana(bk, D, torch.float32)
        prop = bk.CudaProposal(MALA_G, D, params=_mala_params(0.2), gradient=True)
        s = (bk.MetropolisHastings(model, prop, prop.transition_lp, chains=256, seed=1) if hastings
             else bk.Metropolis(model, prop, chains=256, seed=1))
        k0 = _launches()
        s.sample_n(5)
        k1 = _launches()
        s.sample_n(5)
        assert (k1 - k0, _launches() - k1) == (first(5), later(5)), (D, hastings)


def test_errors(bk):
    model = _banana(bk, 3, torch.float32)
    prop = bk.CudaProposal(MALA_G, 3, params=_mala_params(0.2), gradient=True)
    assert "bk_user_propose_grad" in prop.compile_log and "bk_user_dh_grad" in prop.compile_log
    p4 = bk.CudaProposal(MALA_G, 4, params=_mala_params(0.2), gradient=True)
    with pytest.raises(ValueError, match="dims"):
        bk.MetropolisHastings(model, p4, p4.transition_lp)
    p64 = bk.CudaProposal(MALA_G, 3, params=_mala_params(0.2), dtype=torch.float64, gradient=True)
    with pytest.raises(ValueError, match="dims"):
        bk.Metropolis(model, p64)
    # the SMC's move has no gradient form: refused in Python and by the C ABI
    with pytest.raises(ValueError, match="gradient"):
        bk.proposal_kernel(prop)
    pl = bk.CudaPriorLikModel(PRIOR_LIK, 3)
    assert L.lib().bk_smc_cuda_prepare(pl.handle, prop.handle, None, 0) == L.BK_E_UNSUPPORTED
    assert "gradient" in L.lib().bk_last_error().decode()
    # a non-gradient source is not a gradient proposal, and a compile error carries NVRTC's log
    with pytest.raises(ValueError, match="propose"):
        bk.CudaProposal(MALA_G.replace("const bk_real* g, ", ""), 3, params=[0.1, 0.1, 0.1], gradient=True)
    with pytest.raises(ValueError, match=r"proposal.cu\(2\): error"):
        bk.CudaProposal("\n__device__ void propose(const bk_real* t, const bk_real* g, bk_real* q, const bk_real* z, "
                        "const bk_real* u, const bk_real* p) { q[0] = t[0] }", 3, transition=False, gradient=True)
