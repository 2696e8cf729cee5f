"""Stretcher on user-written CUDA models: the fused one-thread-per-walker half-step kernel bk_user_stretch (dims <= 32)
against the oracle, the three-launch engine (BK_FORCE_GENERIC=1), a prior/likelihood restatement and the sharded
ensemble, plus its engine choice, compile errors and statistics."""
import numpy as np
import pytest
import torch

from _dev import np_
from oracle import samplers as osm

pytestmark = pytest.mark.gpu

# ---- models ---------------------------------------------------------------------------------------------------------
# banana: x0 ~ N(0, 1), x1 - b x0^2 ~ N(0, 1), every further coordinate N(0, 1); at D = 1 a standard normal; params = [b]
BANANA = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
#if BK_DIMS == 1
    g[0] = -x[0];
    return bk_real(-0.5) * (x[0] * x[0]);
#else
    const bk_real b = params[0], half = 0.5, two = 2;
    const bk_real u = x[1] - b * x[0] * x[0];
    bk_real lp = -half * (x[0] * x[0]) - half * (u * u);
    g[0] = -x[0] + two * b * x[0] * u;
    g[1] = -u;
    for (int e = 2; e < BK_DIMS; ++e) {
        lp -= half * (x[e] * x[e]);
        g[e] = -x[e];
    }
    return lp;
#endif
}
"""

# non-centred eight schools: theta = (mu, log tau, eta[8]); y_j ~ N(mu + tau eta_j, sigma_j), eta ~ N(0, 1),
# mu ~ N(0, 5^2), log tau ~ N(1, 1); params = [y (8), sigma (8)]
SCHOOLS = """
__device__ bk_real log_density_gradient(const bk_real* th, bk_real* g, const bk_real* p) {
    const bk_real mu = th[0], lt = th[1], tau = exp(lt);
    bk_real lp = -0.5 * (mu * mu) / 25 - 0.5 * ((lt - 1) * (lt - 1));
    bk_real gmu = -mu / 25, glt = -(lt - 1);
    for (int j = 0; j < 8; ++j) {
        const bk_real eta = th[2 + j];
        const bk_real d = p[j] - mu - tau * eta;
        const bk_real r = d / (p[8 + j] * p[8 + j]);
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
SCHOOLS_Y = np.array([28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0])
SCHOOLS_SIGMA = np.array([15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0])

# the banana split into a prior (x0 and x2.. standard normal) and a likelihood (x1 - b x0^2 standard normal), once as
# a CudaPriorLikModel and once as a CudaModel that sums the two terms in the library's order (ll + prior)
BANANA_TERMS = """
__device__ bk_real banana_prior(const bk_real* x, bk_real* g) {
    bk_real s = x[0] * x[0];
    g[0] = -x[0];
    g[1] = 0;
    for (int e = 2; e < BK_DIMS; ++e) {
        s += x[e] * x[e];
        g[e] = -x[e];
    }
    return bk_real(-0.5) * s;
}
__device__ bk_real banana_lik(const bk_real* x, bk_real* g, const bk_real* params) {
    const bk_real b = params[0];
    const bk_real u = x[1] - b * x[0] * x[0];
    for (int e = 0; e < BK_DIMS; ++e) g[e] = 0;
    g[0] = 2 * b * x[0] * u;
    g[1] = -u;
    return bk_real(-0.5) * (u * u);
}
"""
BANANA_PL = BANANA_TERMS + """
__device__ bk_real log_prior_gradient(const bk_real* x, bk_real* g, const bk_real* p) { return banana_prior(x, g); }
__device__ bk_real log_likelihood_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    return banana_lik(x, g, p);
}
"""
BANANA_SUM = BANANA_TERMS + """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real gp[BK_DIMS];
    const bk_real pr = banana_prior(x, gp);
    const bk_real ll = banana_lik(x, g, p);
    for (int e = 0; e < BK_DIMS; ++e) g[e] += gp[e];
    return ll + pr;
}
"""


class NpBanana:
    def __init__(self, D, b):
        self.D, self.b = D, b

    def log_density(self, x):
        x = np.asarray(x, dtype=np.float64)
        if self.D == 1:
            return -0.5 * x[0] * x[0]
        u = x[1] - self.b * x[0] * x[0]
        lp = -0.5 * (x[0] * x[0]) - 0.5 * (u * u)
        for e in range(2, self.D):
            lp -= 0.5 * (x[e] * x[e])
        return lp


class NpSchools:
    def log_density(self, th):
        th = np.asarray(th, dtype=np.float64)
        mu, lt = th[0], th[1]
        tau = np.exp(lt)
        lp = -0.5 * (mu * mu) / 25 - 0.5 * ((lt - 1) * (lt - 1))
        for j in range(8):
            eta = th[2 + j]
            d = SCHOOLS_Y[j] - mu - tau * eta
            r = d / (SCHOOLS_SIGMA[j] * SCHOOLS_SIGMA[j])
            lp += -0.5 * (eta * eta) - 0.5 * (d * r)
        return lp


@pytest.fixture
def fused(monkeypatch):
    monkeypatch.setenv("BK_FORCE_GENERIC", "0")


def _models(bk, which, D, dtype=torch.float64):
    if which == "banana":
        return bk.CudaModel(BANANA, D, params=[0.5], dtype=dtype), NpBanana(D, 0.5)
    return bk.CudaModel(SCHOOLS, 10, params=np.concatenate([SCHOOLS_Y, SCHOOLS_SIGMA]), dtype=dtype), NpSchools()


# ---- 1. oracle parity, fp64, injected uniforms ----------------------------------------------------------------------
@pytest.mark.parametrize("W", [2, 16, 26])
@pytest.mark.parametrize("which,D", [("banana", 1), ("banana", 3), ("banana", 8), ("banana", 32), ("schools", 10)])
def test_matches_oracle(bk, fused, which, D, W):
    n = 6
    dm, om = _models(bk, which, D)
    rng = np.random.default_rng(10 * D + W)
    th0, us = rng.normal(size=(W, D)) * 0.7, rng.random((n, W, 3))
    want, wacc = osm.stretch(om, th0, us, a=2.0)
    s = bk.Stretcher(dm, a=2.0, walkers=W, init=th0)
    assert "bk_user_stretch" in s.compile_log
    for t in range(n):
        got = s.sample(uniforms=us[t])
        assert np.array_equal(np_(s.last_accept).astype(bool), wacc[t]), t
        np.testing.assert_allclose(np_(got), want[t], rtol=1e-10, atol=1e-10)
    assert wacc.any()


# ---- 2. fused == three-launch engine, Philox ------------------------------------------------------------------------
def _pair(bk, monkeypatch, dtype, D=6, W=64):
    monkeypatch.setenv("BK_FORCE_GENERIC", "0")
    dm = bk.CudaModel(BANANA, D, params=[0.5], dtype=dtype)
    init = np.random.default_rng(4).normal(size=(W, D))
    fu = bk.Stretcher(dm, walkers=W, init=init, seed=21)
    ge = bk.Stretcher(dm, walkers=W, init=init, seed=21)
    assert "bk_user_stretch" in fu.compile_log
    return fu, ge


def _sweep(s, monkeypatch, generic):
    """one sample() on the engine BK_FORCE_GENERIC selects at each call"""
    monkeypatch.setenv("BK_FORCE_GENERIC", "1" if generic else "0")
    return s.sample().clone(), s.last_accept.clone()


def test_fused_equals_generic_fp64(bk, monkeypatch):
    """Same uniforms, same Ar<double> operations, the same NVRTC-compiled density: bit for bit."""
    fu, ge = _pair(bk, monkeypatch, torch.float64)
    accs = []
    for t in range(20):
        tf, af = _sweep(fu, monkeypatch, False)
        tg, ag = _sweep(ge, monkeypatch, True)
        assert torch.equal(af, ag), t
        assert torch.equal(tf, tg), t
        assert all(torch.equal(a, b) for a, b in zip(fu._lp, ge._lp)), t
        accs.append(float(af.float().mean()))
    assert 0 < np.mean(accs) < 1


def test_fused_equals_generic_fp32(bk, monkeypatch):
    fu, ge = _pair(bk, monkeypatch, torch.float32)
    for t in range(10):
        tf, af = _sweep(fu, monkeypatch, False)
        tg, ag = _sweep(ge, monkeypatch, True)
        assert torch.equal(af, ag), t
        np.testing.assert_allclose(np_(tf), np_(tg), rtol=1e-6, atol=1e-6)


# ---- 3. engine switch mid-run: the lp cache each engine leaves is valid for the other -------------------------------
@pytest.mark.parametrize("order", ["fused_then_generic", "generic_then_fused"])
def test_engine_switch_mid_run(bk, monkeypatch, order):
    fu, ge = _pair(bk, monkeypatch, torch.float64, D=5, W=40)
    first_generic = order == "generic_then_fused"
    for t in range(12):
        tf, af = _sweep(fu, monkeypatch, first_generic if t < 6 else not first_generic)
        tg, ag = _sweep(ge, monkeypatch, True)
        assert torch.equal(af, ag), t
        assert torch.equal(tf, tg), t


# ---- 4. sharded ensemble ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_equals_oracle(bk, fused, world):
    """Walkers of both halves sharded over `world` ranks of one device, each rank's half-steps on the fused kernel with
    its slice of the injected uniforms: the single-process oracle run."""
    rng = np.random.default_rng(9)
    D, W, n = 7, 26, 5
    dm, om = _models(bk, "banana", D)
    th0 = rng.normal(size=(W, D))
    us = rng.random((n, W, 3))
    want, wacc = osm.stretch(om, th0, us, a=2.0)
    fw = bk.peer.FakeWorld(world)
    ranks = [bk.Stretcher(dm, a=2.0, walkers=W, init=th0, group=fw.rank(r)) for r in range(world)]
    assert all("bk_user_stretch" in s.compile_log for s in ranks)
    h = W // 2
    for t in range(n):
        for half in (0, 1):
            for s in ranks:
                u_loc = np.concatenate([us[t, s._lo:s._hi], us[t, h + s._lo:h + s._hi]])
                s._half_step(half, u_loc)
        torch.cuda.synchronize()
        first = np.concatenate([np_(s._halves[0]) for s in ranks])
        second = np.concatenate([np_(s._halves[1]) for s in ranks])
        np.testing.assert_allclose(np.concatenate([first, second]), want[t], rtol=1e-10, atol=1e-10)
        acc = np.concatenate([np_(s.last_accept).reshape(2, -1)[0] for s in ranks] +
                             [np_(s.last_accept).reshape(2, -1)[1] for s in ranks]).astype(bool)
        assert np.array_equal(acc, wacc[t])


# ---- 5. prior/likelihood models ---------------------------------------------------------------------------------------
def test_prior_lik_equals_model(bk, fused):
    D, W = 6, 64
    pl = bk.CudaPriorLikModel(BANANA_PL, D, params=[0.5], dtype=torch.float64)
    plain = bk.CudaModel(BANANA_SUM, D, params=[0.5], dtype=torch.float64)
    init = np.random.default_rng(6).normal(size=(W, D))
    a = bk.Stretcher(pl, walkers=W, init=init, seed=3)
    b = bk.Stretcher(plain, walkers=W, init=init, seed=3)
    assert "bk_user_stretch" in a.compile_log and "bk_user_stretch" in b.compile_log
    for t in range(10):
        ta, tb = a.sample(), b.sample()
        assert torch.equal(a.last_accept, b.last_accept), t
        assert torch.equal(ta, tb), t
    assert 0 < float(a.last_accept.float().mean()) < 1


# ---- 6. engine choice and surface -------------------------------------------------------------------------------------
def test_engine_choice_and_surface(bk, fused):
    lib = bk._lib.lib()
    for D, want_fused in ((32, True), (33, False)):
        dm = bk.CudaModel(BANANA, D, params=[0.5])
        model_log = dm.compile_log
        s = bk.Stretcher(dm, seed=1)
        assert dm.compile_log == model_log
        assert "bk_user_stretch" not in model_log
        if want_fused:
            assert "Function properties for bk_user_stretch" in s.compile_log
            assert lib.bk_stretch_workspace_bytes(dm.handle, D) == 0
        else:
            assert s.compile_log == ""
        counts = []
        for _ in range(3):
            n0 = lib.bk_launch_count()
            s.sample()
            torch.cuda.synchronize()
            counts.append(lib.bk_launch_count() - n0)
        # three-launch engine: propose, density, accept per half-step, plus the density of the walkers the first time
        assert counts == ([2, 2, 2] if want_fused else [8, 6, 6]), counts


# ---- 7. compile errors -------------------------------------------------------------------------------------------------
def test_compile_error_raises_value_error(bk, fused):
    # compiles as a model; its Stretcher program (-DBK_STRETCH=1) does not
    src = "#ifdef BK_STRETCH\n#error no stretch for this model\n#endif\n" + BANANA
    dm = bk.CudaModel(src, 3, params=[0.5])
    with pytest.raises(ValueError, match="no stretch for this model") as e:
        bk.Stretcher(dm)
    assert str(e.value).startswith("Stretcher: NVRTC compilation of the model's stretch kernel failed:\n")


# ---- 8. statistics, fp32 -----------------------------------------------------------------------------------------------
def test_banana_moments(bk, fused):
    """x1 has mean b and variance 1 + 2 b^2, every other coordinate is N(0, 1); within 4 MCSE (each walker's ESS from
    its own series, summed over walkers)."""
    b, D = 0.5, 8
    dm = bk.CudaModel(BANANA, D, params=[b])
    s = bk.Stretcher(dm, walkers=4096, seed=5)
    assert "bk_user_stretch" in s.compile_log
    for _ in range(500):
        s.sample()
    assert 0.2 < float(s.last_accept.float().mean()) < 0.9
    x = s.sample_n(1000).double()
    mean_t = torch.zeros(D, dtype=torch.float64, device=x.device)
    var_t = torch.ones(D, dtype=torch.float64, device=x.device)
    mean_t[1], var_t[1] = b, 1 + 2 * b * b
    for stat, want in ((x, mean_t), ((x - mean_t) ** 2, var_t)):
        ess = bk.ess(stat, draws_first=True).reshape(-1, D).sum(0)
        est = stat.mean((0, 1))
        mcse = stat.reshape(-1, D).std(0) / ess.sqrt()
        z = ((est - want) / mcse).abs()
        assert float(z.max()) < 4, (np_(est), np_(mcse))
