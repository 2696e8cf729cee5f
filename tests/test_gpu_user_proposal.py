"""CudaProposal: user-written CUDA proposals for Metropolis / MetropolisHastings, compiled at run time.  Each proposal is
written twice, in CUDA for the device and in NumPy for the oracle.  Engines: the fused bk_user_mhp (a user model with
dims <= 32, compiled together with the proposal) and the three-launch path (bk_user_propose, the model's evaluation,
the accept test) for every other model."""
import numpy as np
import pytest
import torch

from _dev import np_
from _user_cuda import (BANANA, DIAG, INDEP, LOGNORMAL, MIXTURE_WALK, RSCAN, RW, NpBanana, check, np_indep,
                        np_lognormal, np_rscan, philox_streams)
from bayes_kit_b200 import _lib as L
from oracle import models as om
from oracle import proposals as opr

pytestmark = pytest.mark.gpu

# ---- models ----------------------------------------------------------------------------------------------------
# independent Gamma(a_e, rate b_e) coordinates, params = [a (D), b (D)].  Its helper `sq` has the name of the log-normal
# proposal's: each source is compiled in a namespace of its own.
GAMMA = """
__device__ bk_real sq(bk_real x) { return x * x; }
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real lp = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        if (!(x[e] > 0)) return log(bk_real(0));
        lp += (p[e] - 1) * log(x[e]) - p[BK_DIMS + e] * x[e];
        g[e] = (p[e] - 1) / x[e] - p[BK_DIMS + e];
    }
    return lp;
}
"""


def _user(bk, src, D, params, dtype=torch.float64):
    return bk.CudaModel(src, D, params=params, dtype=dtype)


def _builtin(bk, kind, D, dtype=torch.float64):
    """(device model, NumPy model) of a built-in plugin."""
    rng = np.random.default_rng(D)
    if kind == "diag":
        mu, pr = rng.normal(size=D), rng.uniform(0.5, 3.0, D)
        return bk.DiagGauss(mu, pr, dtype=dtype), om.DiagGauss(mu, pr)
    if kind == "dense":
        P = om.DensePrecGauss.c2_precision(D, 1)
        return bk.DensePrecGauss(P, dtype=dtype), om.DensePrecGauss(P)
    if kind == "binom":
        return bk.Binomial(2.0, 3.0, 7, 20, dtype=dtype), om.Binomial(2.0, 3.0, 7, 20)
    if kind == "hlr":
        X, y = om.HierLogReg.c3_data(50, D - 2, seed=2)
        return bk.HierLogReg(X, y, dtype=dtype), om.HierLogReg(X, y)
    raise ValueError(kind)


def _launches(bk):
    return int(L.lib().bk_launch_count())


# ---- 1. the random walk restated equals the built-in -----------------------------------------------------------------
def _pair(bk, model, D, s, init, dtype, seed=5):
    prop = bk.CudaProposal(RW, D, params=[s], dtype=dtype)
    return (bk.Metropolis(model, prop, init=init, seed=seed), bk.Metropolis(model, bk.GaussianRW(s), init=init, seed=seed))


def _same_run(a, b, n, injected, dtype, exact=True):
    C_, D = a.chains, a._dim
    kw = {}
    if injected:
        rng = np.random.default_rng(D + C_)
        kw = dict(normals=rng.standard_normal((n, C_, D)), uniforms=rng.random((n, C_, 1)))
    da, la = a.sample_n(n, **kw)
    db, lb = b.sample_n(n, **kw)
    assert torch.equal(a.last_accept, b.last_accept)
    assert 0 < float(a.last_accept.float().mean()) < 1
    if exact:
        assert torch.equal(da, db) and torch.equal(la, lb)
    else:
        np.testing.assert_allclose(np_(da), np_(db), rtol=1e-5, atol=1e-5)


# NVRTC and nvcc both contract theta + s * z into one FMA in fp32 (neither is given --fmad=false there), so the fp32 runs
# are compared bit for bit too.
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("injected", [False, True])
@pytest.mark.parametrize("D", [2, 17, 32, 40, 100])
def test_restated_rw_equals_builtin_user_model(bk, D, injected, dtype):
    """D <= 32: bk_user_mhp against bk_user_mh; D = 40, 100: the three-launch path against the generic engine."""
    model = _user(bk, BANANA, D, [0.5], dtype)
    init = np.random.default_rng(D).normal(size=(70, D))
    a, b = _pair(bk, model, D, 1.2 / np.sqrt(D), init, dtype)
    _same_run(a, b, 8, injected, dtype)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("injected", [False, True])
@pytest.mark.parametrize("kind,D", [("diag", 7), ("dense", 50), ("binom", 1)])
def test_restated_rw_equals_builtin_plugins(bk, monkeypatch, kind, D, injected, dtype):
    monkeypatch.setenv("BK_FORCE_GENERIC", "1")
    model, _ = _builtin(bk, kind, D, dtype)
    init = np.random.default_rng(3).normal(size=(45, D))
    a, b = _pair(bk, model, D, 1.0 / np.sqrt(D), init, dtype)
    _same_run(a, b, 8, injected, dtype)


# ---- 2. oracle parity under injected streams, fp64 -------------------------------------------------------------------
def _proposal(bk, which, D):
    if which == "indep":
        rng = np.random.default_rng(40 + D)
        m, s = rng.normal(size=D) * 0.3, rng.uniform(0.7, 1.5, D)
        return bk.CudaProposal(INDEP, D, params=np.concatenate([m, s]), dtype=torch.float64), np_indep(m, s), True
    if which == "lognormal":
        return bk.CudaProposal(LOGNORMAL, D, params=[0.3], dtype=torch.float64), np_lognormal(0.3), True
    return (bk.CudaProposal(RSCAN, D, params=[0.8], normals=1, uniforms=1, dtype=torch.float64), np_rscan(0.8),
            False)


MODELS = [("user", 3), ("user", 40), ("diag", 6), ("dense", 8), ("hlr", 6)]


@pytest.mark.parametrize("which", ["indep", "lognormal", "rscan"])
@pytest.mark.parametrize("mk", range(len(MODELS)))
def test_matches_oracle(bk, which, mk):
    kind, D = MODELS[mk]
    C_ = (1, 37, 129)[(mk + len(which)) % 3]
    n = 6
    if kind == "user":
        dev, npm = _user(bk, BANANA, D, [0.5]), NpBanana(D, 0.5)
    else:
        dev, npm = _builtin(bk, kind, D)
    prop, (propose, tld), asym = _proposal(bk, which, D)
    rng = np.random.default_rng(mk * 10 + len(which))
    th0 = rng.normal(size=(C_, D)) * 0.5
    if which == "lognormal":
        th0 = np.abs(th0) + 0.2
    zs = rng.standard_normal((n, C_, prop.normals))
    us = rng.random((n, C_, 1 + prop.uniforms))
    s = bk.MetropolisHastings(dev, prop, prop.transition_lp, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    check(d, l, s.last_accept, opr.metropolis_hastings_batch(npm, th0, zs, us, propose, tld))
    if not asym:
        s = bk.Metropolis(dev, prop, init=th0)
        d, l = s.sample_n(n, normals=zs, uniforms=us)
        check(d, l, s.last_accept, opr.metropolis_hastings_batch(npm, th0, zs, us, propose))


# ---- 3. Philox equals the injected reconstruction (fp64) -------------------------------------------------------------
@pytest.mark.parametrize("offset", [0, 1000])
@pytest.mark.parametrize("engine", ["fused", "three-launch"])
@pytest.mark.parametrize("which", ["mixture", "rscan", "rw"])
def test_philox_equals_injected_reconstruction(bk, which, engine, offset):
    D, C_, n, seed = 5, 33, 5, 77
    if engine == "fused":
        model = _user(bk, BANANA, D, [0.5])
    else:
        model = _builtin(bk, "diag", D)[0]
    if which == "mixture":
        prop = bk.CudaProposal(MIXTURE_WALK, D, params=[0.3, 1.5, 0.4], normals=2 * D, uniforms=2, transition=False,
                               dtype=torch.float64)
    elif which == "rscan":
        prop = bk.CudaProposal(RSCAN, D, params=[0.8], normals=1, uniforms=1, dtype=torch.float64)
    else:
        prop = bk.CudaProposal(RW, D, params=[0.7], dtype=torch.float64)
    init = np.random.default_rng(1).normal(size=(C_, D))
    a = bk.Metropolis(model, prop, init=init, seed=seed, chain_offset=offset)
    b = bk.Metropolis(model, prop, init=init, seed=seed, chain_offset=offset)
    Z, U = philox_streams(bk, seed, offset, C_, D, prop.normals, prop.uniforms, n, 0)
    da, la = a.sample_n(n)
    db, lb = b.sample_n(n, normals=Z, uniforms=U)
    assert torch.equal(a.last_accept, b.last_accept)
    assert 0 < float(a.last_accept.float().mean()) < 1
    assert torch.equal(da, db) and torch.equal(la, lb)


# ---- 4. statistics, fp32 Philox ---------------------------------------------------------------------------------------
def _z_scores(bk, x, want):
    D = x.shape[-1]
    ess = bk.ess(x, draws_first=True).reshape(-1, D).sum(0)
    est = x.mean((0, 1))
    mcse = x.reshape(-1, D).std(0) / ess.sqrt()
    return ((est - want) / mcse).abs(), est


def test_lognormal_walk_needs_the_hastings_term(bk):
    """Gamma(a, b) coordinates: mean a / b, variance a / b^2.  Without the Hastings term (Metropolis) the walk samples
    Gamma(a - 1, b) instead -- it must miss the mean by far."""
    a_, b_ = np.array([2.0, 3.0, 4.0, 5.0]), np.array([1.0, 2.0, 1.5, 3.0])
    model = bk.CudaModel(GAMMA, 4, params=np.concatenate([a_, b_]))
    prop = bk.CudaProposal(LOGNORMAL, 4, params=[0.5])
    init = (a_ / b_) * np.exp(0.3 * np.random.default_rng(0).normal(size=(4096, 4)))
    mean_t = torch.tensor(a_ / b_, device="cuda")
    var_t = torch.tensor(a_ / b_ ** 2, device="cuda")
    s = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init, seed=21)
    s.sample_n(300, keep_draws=False)
    x = s.sample_n(300)[0].double()
    zm, est = _z_scores(bk, x, mean_t)
    zv, _ = _z_scores(bk, (x - mean_t) ** 2, var_t)
    assert float(zm.max()) < 4 and float(zv.max()) < 4, (np_(est), np_(zm), np_(zv))
    s = bk.Metropolis(model, prop, init=init, seed=21)
    s.sample_n(300, keep_draws=False)
    zm, est = _z_scores(bk, s.sample_n(300)[0].double(), mean_t)
    assert float(zm.min()) > 10, (np_(est), np_(zm))


def test_exact_independence_sampler_accepts_everything(bk):
    mu, sd = np.array([0.5, -1.0, 2.0]), np.array([1.0, 0.5, 2.0])
    model = bk.CudaModel(DIAG, 3, params=np.concatenate([mu, 1 / sd ** 2]))
    prop = bk.CudaProposal(INDEP, 3, params=np.concatenate([mu, sd]))
    s = bk.MetropolisHastings(model, prop, prop.transition_lp, chains=2048, seed=3)
    s.sample_n(50)
    assert float(s.last_accept.float().mean()) >= 0.999


# ---- 5. shard invariance ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [6, 40])
def test_shards_equal_one_sampler(bk, D):
    model = _user(bk, BANANA, D, [0.5], torch.float32)
    prop = bk.CudaProposal(RSCAN, D, params=[0.9], normals=1, uniforms=1)
    init = np.random.default_rng(D).normal(size=(96, D))
    full = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init, seed=4).sample_n(10)[0]
    lo = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init[:40], seed=4).sample_n(10)[0]
    hi = bk.MetropolisHastings(model, prop, prop.transition_lp, init=init[40:], seed=4, chain_offset=40).sample_n(10)[0]
    assert torch.equal(full, torch.cat([lo, hi], 1))


# ---- 6. plumbing ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["user8", "user40", "diag"])
def test_host_draws_moments_and_layout(bk, kind):
    if kind == "diag":
        model = _builtin(bk, "diag", 12, torch.float32)[0]
    else:
        model = _user(bk, BANANA, int(kind[4:]), [0.5], torch.float32)
    D = model.dims()
    prop = bk.CudaProposal(RW, D, params=[0.5])
    make = lambda: bk.MetropolisHastings(model, prop, prop.transition_lp, chains=300, seed=8)   # noqa: E731
    a, b, c = make(), make(), make()
    da, la = a.sample_n(5)
    hd, hl = b.sample_host_n(5)
    assert torch.equal(da.cpu(), hd) and torch.equal(la.cpu(), hl)
    h1, l1 = c.sample_host()
    assert torch.equal(da[0].cpu(), h1) and torch.equal(la[0].cpu(), l1)
    s = make()
    d1, _ = s.sample_n(9, moments=True)
    d2, _ = s.sample_n(7, moments=True)
    mean, var, n = s.running_moments()
    x = torch.cat([d1, d2]).double()
    assert n == 16
    np.testing.assert_allclose(np_(mean), np_(x.mean(0)), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(np_(var), np_(x.var(0)), rtol=1e-7, atol=1e-9)
    with pytest.raises(NotImplementedError, match="series"):
        s.sample_n(3, layout="series")


def test_launch_counts_show_the_engine(bk):
    for D, per_call in ((8, lambda n: 1), (40, lambda n: 3 * n + 1)):
        model = _user(bk, BANANA, D, [0.5], torch.float32)
        prop = bk.CudaProposal(RW, D, params=[0.5])
        s = bk.MetropolisHastings(model, prop, prop.transition_lp, chains=256, seed=1)
        k0 = _launches(bk)
        s.sample_n(5)
        assert _launches(bk) - k0 == per_call(5), D


# ---- 7. errors --------------------------------------------------------------------------------------------------------
def test_errors(bk):
    model = _user(bk, BANANA, 3, [0.5], torch.float32)
    with pytest.raises(ValueError, match="dims"):
        bk.Metropolis(model, bk.CudaProposal(RW, 4, params=[0.5]))
    with pytest.raises(ValueError, match="dims"):
        bk.Metropolis(model, bk.CudaProposal(RW, 3, params=[0.5], dtype=torch.float64))
    sym = bk.CudaProposal(MIXTURE_WALK, 3, params=[0.3, 1.5, 0.4], normals=6, uniforms=2, transition=False)
    bk.Metropolis(model, sym)
    with pytest.raises(TypeError, match="transition"):
        bk.MetropolisHastings(model, sym, sym.transition_lp)
    prop = bk.CudaProposal(RW, 3, params=[0.5])
    with pytest.raises(TypeError, match="transition_lp_fn"):
        bk.MetropolisHastings(model, prop, bk.CudaProposal(RW, 3, params=[0.5]).transition_lp)
    with pytest.raises(TypeError, match="transition_lp_fn"):
        bk.MetropolisHastings(model, prop, lambda to, frm: 0.0)
    with pytest.raises(TypeError, match="proposal descriptor"):
        bk.MetropolisHastings(model, lambda x: x, prop.transition_lp)
    with pytest.raises(TypeError, match="device-side descriptor"):
        prop.transition_lp(None, None)
    with pytest.raises(ValueError, match=r'proposal.cu\(2\): error'):
        bk.CudaProposal("\n__device__ void propose(const bk_real* t, bk_real* q, const bk_real* z, const bk_real* u, "
                        "const bk_real* p) { q[0] = t[0] }", 3, transition=False)
    assert "bk_user_propose" in prop.compile_log
    # the C entry point refuses a proposal handle where a model handle belongs, and a foreign uniform count
    assert L.lib().bk_model_dims(prop.handle) == -1
    s = bk.Metropolis(model, sym, chains=4)
    with pytest.raises(ValueError, match="n_uniform"):
        s._n_uniform = 1
        s.sample_n(1, normals=np.zeros((1, 4, 6)), uniforms=np.full((1, 4, 1), 0.5))
