"""CudaModel: user-written CUDA log densities compiled at run time.  Each model is written twice, in CUDA for the
device and in NumPy for the oracle.  Parity runs fp64 with injected streams on both engines (the fused one-thread-
per-chain kernels and, with BK_FORCE_GENERIC=1, the generic engine through bk_user_eval)."""
import numpy as np
import pytest
import torch

from _dev import np_
from _user_cuda import (BANANA, DIAG, SCHOOLS_SIGMA, SCHOOLS_Y, NpSchools, banana, check, diag_params,
                        streams_uniforms_first)
from oracle import samplers as osm
from oracle.models import DiagGauss as ODiag

pytestmark = pytest.mark.gpu

# ---- models ----------------------------------------------------------------------------------------------------
# non-centred eight schools: theta = (mu, log tau, eta[8]); y_j ~ N(mu + tau eta_j, sigma_j), eta ~ N(0, 1),
# mu ~ N(0, 5^2), log tau ~ N(1, 1); params = [y (8), sigma (8)]
SCHOOLS = """
struct School { bk_real y, sigma; };
__device__ School school(const bk_real* p, int j) { return School{p[j], p[8 + j]}; }

__device__ bk_real log_density_gradient(const bk_real* th, bk_real* g, const bk_real* p) {
    const bk_real mu = th[0], lt = th[1], tau = exp(lt);
    bk_real lp = -0.5 * (mu * mu) / 25 - 0.5 * ((lt - 1) * (lt - 1));
    bk_real gmu = -mu / 25, glt = -(lt - 1);
    for (int j = 0; j < 8; ++j) {
        const School s = school(p, j);
        const bk_real eta = th[2 + j];
        const bk_real d = s.y - mu - tau * eta;
        const bk_real r = d / (s.sigma * s.sigma);
        lp += -0.5 * (eta * eta) - 0.5 * (d * r);
        gmu += r;
        glt += r * tau * eta;
        g[2 + j] = -eta + r * tau;
    }
    g[0] = gmu;
    g[1] = glt;
    return lp;
}
"""


@pytest.fixture(params=["fused", "generic"])
def engine(request, monkeypatch):
    monkeypatch.setenv("BK_FORCE_GENERIC", "1" if request.param == "generic" else "0")
    return request.param


# ---- 1. protocol ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["banana", "diag", "schools"])
def test_protocol_matches_numpy(bk, which):
    rng = np.random.default_rng(1)
    if which == "banana":
        dm, om = banana(bk, 5)
    elif which == "diag":
        mu, pr = diag_params(7)
        dm, om = bk.CudaModel(DIAG, 7, params=np.concatenate([mu, pr]), dtype=torch.float64), ODiag(mu, pr)
    else:
        dm = bk.CudaModel(SCHOOLS, 10, params=np.concatenate([SCHOOLS_Y, SCHOOLS_SIGMA]), dtype=torch.float64)
        om = NpSchools()
    D = dm.dims()
    X = rng.normal(size=(33, D))
    lp, g = dm.log_density_gradient(X)
    want = [om.log_density_gradient(x) for x in X]
    np.testing.assert_allclose(np_(lp), [w[0] for w in want], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(g), np.stack([w[1] for w in want]), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(dm.log_density(X)), [w[0] for w in want], rtol=1e-12, atol=1e-12)
    one = dm.log_density(X[0])
    assert isinstance(one, float) and one == pytest.approx(want[0][0], rel=1e-12)
    l1, g1 = dm.log_density_gradient(X[0])
    assert isinstance(l1, float) and g1.shape == (D,)
    np.testing.assert_allclose(np_(g1), want[0][1], rtol=1e-12, atol=1e-12)


# ---- 2. reference parity ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [0, 1, 7])
@pytest.mark.parametrize("metric", [False, True])
def test_hmc_matches_oracle(bk, engine, L, metric):
    C, D, n = 37, 3, 6
    dm, om = banana(bk, D)
    th0, zs, us = streams_uniforms_first(C, D, n, L)
    m = np.array([1.0, 0.5, 2.0]) if metric else None
    s = bk.HMCDiag(dm, 0.3, L, metric_diag=m, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    check(d, l, s.last_accept, osm.hmc_diag_batch(om, th0, zs, us, 0.3, L, m))
    np.testing.assert_allclose(np_(s.theta), np_(d[-1]), rtol=0, atol=0)


def test_mala_matches_oracle(bk, engine):
    C, D, n = 37, 4, 6
    dm, om = banana(bk, D)
    th0, zs, us = streams_uniforms_first(C, D, n, 11)
    s = bk.MALA(dm, 0.2, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    check(d, l, s.last_accept, osm.mala_batch(om, th0, zs, us, 0.2))


@pytest.mark.parametrize("hastings", [False, True])
def test_metropolis_matches_oracle(bk, engine, hastings):
    C, D, n = 37, 5, 6
    dm, om = banana(bk, D)
    th0, zs, us = streams_uniforms_first(C, D, n, 12)
    prop = bk.GaussianRW(0.6)
    s = bk.MetropolisHastings(dm, prop, prop.transition_lp, init=th0) if hastings else bk.Metropolis(dm, prop, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    check(d, l, s.last_accept, osm.metropolis_rw_batch(om, th0, zs, us, 0.6, hastings))


def test_schools_hmc_matches_oracle(bk, engine):
    C, D, n = 19, 10, 4
    dm = bk.CudaModel(SCHOOLS, 10, params=np.concatenate([SCHOOLS_Y, SCHOOLS_SIGMA]), dtype=torch.float64)
    th0, zs, us = streams_uniforms_first(C, D, n, 13)
    s = bk.HMCDiag(dm, 0.1, 5, init=th0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    check(d, l, s.last_accept, osm.hmc_diag_batch(NpSchools(), th0, zs, us, 0.1, 5))


@pytest.mark.parametrize("K", [2, 3])
def test_drghmc_matches_oracle(bk, K):
    C, D, n = 23, 3, 5
    dm, om = banana(bk, D)
    th0, zs, us = streams_uniforms_first(C, D, n, 20 + K, n_uniform=2 * K)
    rho0 = np.random.default_rng(K).normal(size=(C, D))
    sizes, counts = [0.4, 0.2, 0.1][:K], [2, 4, 8][:K]
    s = bk.DrGhmcDiag(dm, K, sizes, counts, 0.5, init=th0)
    s.set_momentum(rho0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    wd, wl, wrho, wused = osm.drghmc_batch(om, th0, rho0, zs, us, K, sizes, counts, 0.5)[:4]
    assert np.array_equal(np_(s.last_n_uniform), wused)
    np.testing.assert_allclose(np_(d), wd, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(np_(l), wl, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(np_(s.rho), wrho, rtol=1e-10, atol=1e-10)


def test_stretcher_matches_oracle(bk):
    W, D, n = 16, 3, 6
    dm, om = banana(bk, D)
    rng = np.random.default_rng(5)
    th0, us = rng.normal(size=(W, D)), rng.random((n, W, 3))
    want, wacc = osm.stretch(om, th0, us, a=2.0)
    s = bk.Stretcher(dm, a=2.0, walkers=W, init=th0)
    for t in range(n):
        got = s.sample(uniforms=us[t])
        assert np.array_equal(np_(s.last_accept).astype(bool), wacc[t])
        np.testing.assert_allclose(np_(got), want[t], rtol=1e-10, atol=1e-10)


# ---- 3. same RNG as the built-in plugins ---------------------------------------------------------------------------
@pytest.mark.parametrize("D", [3, 8])
def test_user_diag_gauss_equals_builtin(bk, D):
    mu, pr = diag_params(D)
    user = bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]), dtype=torch.float64)
    built = bk.DiagGauss(mu, pr, dtype=torch.float64)
    init = np.random.default_rng(D).normal(size=(64, D))
    for make in (lambda m: bk.HMCDiag(m, 0.3, 4, init=init, seed=17),
                 lambda m: bk.MALA(m, 0.1, init=init, seed=17),
                 lambda m: bk.Metropolis(m, bk.GaussianRW(0.5), init=init, seed=17)):
        a, b = make(user), make(built)
        da, la = a.sample_n(20)
        db, lb = b.sample_n(20)
        assert torch.equal(a.last_accept, b.last_accept)
        assert 0 < float(a.last_accept.float().mean()) < 1
        np.testing.assert_allclose(np_(da), np_(db), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(np_(la), np_(lb), rtol=1e-12, atol=1e-12)


def test_fused_equals_generic_and_shard_invariant(bk, monkeypatch):
    dm, _ = banana(bk, 6)
    init = np.random.default_rng(2).normal(size=(64, 6))
    out = {}
    for eng in ("0", "1"):
        monkeypatch.setenv("BK_FORCE_GENERIC", eng)
        s = bk.HMCDiag(dm, 0.25, 5, init=init, seed=9)
        out[eng] = (s.sample_n(20), s.last_accept)
    assert torch.equal(out["0"][1], out["1"][1])
    np.testing.assert_allclose(np_(out["0"][0][0]), np_(out["1"][0][0]), rtol=1e-12, atol=1e-12)
    monkeypatch.setenv("BK_FORCE_GENERIC", "0")
    full = bk.HMCDiag(dm, 0.25, 5, init=init, seed=9).sample_n(10)[0]
    part = bk.HMCDiag(dm, 0.25, 5, init=init[40:64], seed=9, chain_offset=40).sample_n(10)[0]
    assert torch.equal(full[:, 40:64], part)


# ---- 4. statistics, fp32 -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [8, 100])
def test_banana_moments(bk, D):
    """Closed-form moments: x1 has mean b and variance 1 + 2 b^2, every other coordinate is N(0, 1).  D = 8 runs
    the fused kernel, D = 100 the generic engine."""
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
        ess = bk.ess(stat, draws_first=True).reshape(-1, D).sum(0)   # pooled over chains, per dimension
        est = stat.mean((0, 1))
        mcse = stat.reshape(-1, D).std(0) / ess.sqrt()
        z = ((est - want) / mcse).abs()
        assert float(z.max()) < 4, (np_(est), np_(mcse))


# ---- 5. surface and errors -----------------------------------------------------------------------------------------
def test_compile_errors_raise_value_error(bk):
    with pytest.raises(ValueError, match=r'model.cu\(2\): error: expected a ";"'):
        bk.CudaModel("\n__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) "
                     "{ return x[0] }", 2)
    with pytest.raises(ValueError, match="log_density_gradient"):
        bk.CudaModel("__device__ bk_real log_density(const bk_real* x) { return x[0]; }", 2)
    for dims in (0, 65537):
        with pytest.raises(ValueError, match="dims"):
            bk.CudaModel(BANANA, dims, params=[0.5])
    with pytest.raises(TypeError, match="dims"):
        bk.CudaModel(BANANA, 2.0, params=[0.5])
    dm, _ = banana(bk, 2)
    assert "bk_user_hmc" in dm.compile_log
    with pytest.raises(TypeError, match="log_prior/log_likelihood"):
        bk.TemperedLikelihoodSMC(dm, 64, 3, np.zeros((64, 2)), bk.metropolis_kernel(0.3))


@pytest.mark.parametrize("D", [4, 40])
def test_moments_and_host_draws(bk, D):
    dm = bk.CudaModel(BANANA, D, params=[0.5])
    s = bk.HMCDiag(dm, 0.2, 4, chains=256, seed=4)
    d1, _ = s.sample_n(9, moments=True)
    d2, _ = s.sample_n(7, moments=True)
    np.testing.assert_allclose(np_(s.running_rhat()), np_(bk.rhat(torch.cat([d1, d2]), draws_first=True)), rtol=1e-4)
    a = bk.HMCDiag(dm, 0.2, 4, chains=256, seed=4)
    b = bk.HMCDiag(dm, 0.2, 4, chains=256, seed=4)
    da, la = a.sample_n(5)
    hd, hl = b.sample_host_n(5)
    assert torch.equal(da.cpu(), hd) and torch.equal(la.cpu(), hl)
