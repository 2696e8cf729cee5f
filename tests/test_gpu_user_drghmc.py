"""DrGhmcDiag on user-written CUDA models: the fused one-thread-per-chain kernel bk_user_drghmc (dims <= 32) against
the oracle, the reference's golden trajectories, the lockstep engine (BK_FORCE_GENERIC=1) and the built-in plugin's
fused kernel, plus its host surface, statistics and engine choice."""
import numpy as np
import pytest
import torch

from _dev import assert_traj, np_
from conftest import golden
from oracle import samplers as osm
from test_gpu_user_model import BANANA, DIAG, _diag_params
from test_gpu_user_smc import GPL, binom

pytestmark = pytest.mark.gpu

# the banana of test_gpu_user_model.py, also defined at D = 1 (then a standard normal); params = [b]
BANANA_1 = """
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

# a standard normal truncated to x0 >= 0: log p = -inf on half the space
HALF_NORMAL = """
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* params) {
    bk_real s = 0;
    for (int e = 0; e < BK_DIMS; ++e) {
        s += x[e] * x[e];
        g[e] = -x[e];
    }
    return x[0] < 0 ? log(bk_real(0)) : bk_real(-0.5) * s;
}
"""


class NpBanana:
    def __init__(self, D, b):
        self.D, self.b = D, b

    def dims(self):
        return self.D

    def log_density_gradient(self, x):
        x = np.asarray(x, dtype=np.float64)
        if self.D == 1:
            return -0.5 * x[0] * x[0], -x.copy()
        u = x[1] - self.b * x[0] * x[0]
        lp = -0.5 * (x[0] * x[0]) - 0.5 * (u * u)
        g = -x.copy()
        g[0] = -x[0] + 2 * self.b * x[0] * u
        g[1] = -u
        for e in range(2, self.D):
            lp -= 0.5 * (x[e] * x[e])
        return lp, g

    def log_density(self, x):
        return self.log_density_gradient(x)[0]


@pytest.fixture
def fused(monkeypatch):
    monkeypatch.setenv("BK_FORCE_GENERIC", "0")


def _oracle_trace(monkeypatch):
    """Records the oracle's log acceptance probabilities of the proposals made from the chain state, in call order, and
    counts its ghost early exits (a ghost with accept_logp == 0, drghmc.py:430-432)."""
    orig = osm._DrState.log_accept
    st = {"depth": 0, "exits": 0, "top": []}

    def log_accept(self, q, r, k, ch, cl):
        st["depth"] += 1
        try:
            a, lp = orig(self, q, r, k, ch, cl)
        finally:
            st["depth"] -= 1
        if st["depth"] > 0 and a == 0:
            st["exits"] += 1
        if st["depth"] == 0:
            st["top"].append(a)
        return a, lp

    monkeypatch.setattr(osm._DrState, "log_accept", log_accept)
    return st


def _oracle_accepts(trace, used, us):
    """The oracle's accept flags [n, C]: a draw moved iff its last proposal passed its accept test (the position alone
    cannot tell: a trajectory may return to its start).  drghmc_batch runs chain by chain, draw by draw; a draw makes
    used // 2 proposals."""
    n, C = used.shape
    top, i = trace["top"], 0
    acc = np.zeros((n, C), dtype=bool)
    for c in range(C):
        for t in range(n):
            i += used[t, c] // 2
            if used[t, c] % 2 == 0:
                acc[t, c] = osm._log_u(us[t, c, used[t, c] - 1]) < top[i - 1]
    assert i == len(top)
    return acc


# ---- 1. oracle parity, fp64, injected streams ---------------------------------------------------------------------
# step sizes chosen so that every case takes each branch open to it (asserted below); at D = 1 the standard normal
# needs larger steps to be rejected at all
SIZES = [1.3, 0.65, 0.33, 0.17, 0.09, 0.05]
SIZES_D1 = [2.2, 1.9, 1.6, 1.3, 1.0, 0.7]
COUNTS = [2, 3, 4, 5, 6, 7]


@pytest.mark.parametrize("metric", [False, True])
@pytest.mark.parametrize("prob_retry", [True, False])
@pytest.mark.parametrize("K", [1, 2, 3, 6])
@pytest.mark.parametrize("D", [1, 3, 8, 32])
def test_matches_oracle(bk, fused, monkeypatch, D, K, prob_retry, metric):
    C, n = 64, 6
    rng = np.random.default_rng(100 * D + 10 * K + 2 * prob_retry + metric)
    th0, rho0 = rng.normal(size=(C, D)) * 0.7, rng.normal(size=(C, D))
    zs, us = rng.standard_normal((n, C, D)), rng.random((n, C, 2 * K))
    m = np.linspace(0.5, 2.0, D) if metric else None
    sizes, counts = (SIZES_D1 if D == 1 else SIZES)[:K], COUNTS[:K]
    dm = bk.CudaModel(BANANA_1, D, params=[0.5], dtype=torch.float64)
    s = bk.DrGhmcDiag(dm, K, sizes, counts, 0.5, metric_diag=m, init=th0, prob_retry=prob_retry)
    assert "bk_user_drghmc" in s.compile_log
    s.set_momentum(rho0)
    d, l = s.sample_n(n, normals=zs, uniforms=us)
    trace = _oracle_trace(monkeypatch)
    wd, wl, wrho, wused = osm.drghmc_batch(NpBanana(D, 0.5), th0, rho0, zs, us, K, sizes, counts, 0.5, m,
                                           prob_retry)[:4]
    used, acc = np_(s.last_n_uniform), np_(s.last_accept).astype(bool)
    assert np.array_equal(used, wused)
    assert np.array_equal(acc, _oracle_accepts(trace, wused, us))
    np.testing.assert_allclose(np_(d), wd, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(np_(l), wl, rtol=1e-10, atol=1e-10)
    np.testing.assert_allclose(np_(s.rho), wrho, rtol=1e-10, atol=1e-10)
    taken = {"first-proposal accept": np.any(acc & (used == 2)), "later accept": np.any(acc & (used > 2)),
             "all rejected": np.any(~acc & (used == 2 * K)), "retry stop": np.any(used % 2 == 1),
             "ghost early exit": trace["exits"] > 0}
    open_ = {"first-proposal accept": True, "later accept": K >= 2, "all rejected": True,
             "retry stop": K >= 2 and prob_retry, "ghost early exit": K >= 2}
    assert [b for b in taken if open_[b] and not taken[b]] == []


# ---- 2. the reference's golden trajectories through restated models -----------------------------------------------
def _restated(bk, z):
    kind = str(z["model_kind"])
    if kind == "iso":
        D = int(z["model_dims"])
        prec = np.full(D, 1.0 / float(z["model_sigma"]) ** 2)
        return bk.CudaModel(DIAG, D, params=np.concatenate([np.zeros(D), prec]), dtype=torch.float64)
    if kind == "diag":
        return bk.CudaModel(DIAG, len(z["model_mu"]), params=np.concatenate([z["model_mu"], z["model_prec"]]),
                            dtype=torch.float64)
    a, b, x, n = z["model_abxn"]
    return binom(bk, float(a), float(b), int(x), int(n))


@pytest.mark.parametrize("name", ["drghmc_iso_d10_retry0", "drghmc_iso_d10_retry1", "drghmc_diag_d7_k4",
                                  "drghmc_binom"])
def test_golden(bk, fused, name):
    z = golden(name)
    K = int(z["max_proposals"])
    s = bk.DrGhmcDiag(_restated(bk, z), K, [float(v) for v in z["step_sizes"]], [int(v) for v in z["step_counts"]],
                      float(z["damping"]), init=z["theta0"], prob_retry=bool(z["prob_retry"]))
    assert "bk_user_drghmc" in s.compile_log
    s.set_momentum(z["rho0"])
    u = np.nan_to_num(z["uniforms"], nan=0.5)
    draws, logp = s.sample_n(z["normals"].shape[0], normals=z["normals"], uniforms=u)
    assert np.array_equal(np_(s.last_n_uniform), z["n_used"]), "uniform consumption differs"
    assert_traj(draws, logp, s.last_accept, z)
    np.testing.assert_allclose(np_(s.rho), z["rho_final"], rtol=1e-10, atol=1e-10)


# ---- 3. fused == lockstep -----------------------------------------------------------------------------------------
def _both_engines(monkeypatch, make, n=20):
    out = {}
    for eng in ("0", "1"):
        monkeypatch.setenv("BK_FORCE_GENERIC", eng)
        s = make()
        assert ("bk_user_drghmc" in s.compile_log) == (eng == "0")
        d, l = s.sample_n(n)
        out[eng] = (d, l, s.last_accept, s.last_n_uniform, s.rho)
    (d0, l0, a0, u0, r0), (d1, l1, a1, u1, r1) = out["0"], out["1"]
    assert torch.equal(u0, u1) and torch.equal(a0, a1)
    assert 0 < float(a0.float().mean()) < 1
    np.testing.assert_allclose(np_(d0), np_(d1), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(l0), np_(l1), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(r0), np_(r1), rtol=1e-12, atol=1e-12)
    return out


@pytest.mark.parametrize("which", ["model", "prior_lik"])
def test_fused_equals_lockstep(bk, monkeypatch, which):
    rng = np.random.default_rng(7)
    if which == "model":
        D = 6
        dm = bk.CudaModel(BANANA, D, params=[0.5], dtype=torch.float64)
    else:
        D = 5
        m0, p0, mu, pl = rng.normal(size=D), rng.uniform(0.5, 2, D), rng.normal(size=D), rng.uniform(1, 4, D)
        dm = bk.CudaPriorLikModel(GPL, D, params=np.concatenate([mu, pl, m0, p0]), dtype=torch.float64)
    init = rng.normal(size=(64, D))
    _both_engines(monkeypatch, lambda: bk.DrGhmcDiag(dm, 3, [0.9, 0.45, 0.2], [3, 6, 12], 0.5, init=init, seed=11))


def test_minus_inf_region_fused_equals_lockstep(bk, monkeypatch):
    dm = bk.CudaModel(HALF_NORMAL, 4, dtype=torch.float64)
    init = np.abs(np.random.default_rng(8).normal(size=(64, 4)))
    out = _both_engines(monkeypatch, lambda: bk.DrGhmcDiag(dm, 3, [0.8, 0.4, 0.2], [2, 4, 8], 0.5, init=init, seed=5))
    assert float(out["0"][0][..., 0].min()) >= 0


# ---- 4. the built-in plugin's words -------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [3, 8])
def test_user_diag_gauss_equals_builtin(bk, fused, D):
    mu, pr = _diag_params(D)
    user = bk.CudaModel(DIAG, D, params=np.concatenate([mu, pr]), dtype=torch.float64)
    built = bk.DiagGauss(mu, pr, dtype=torch.float64)
    init = np.random.default_rng(D).normal(size=(64, D))
    a = bk.DrGhmcDiag(user, 3, [0.8, 0.4, 0.2], [2, 4, 8], 0.5, init=init, seed=17)
    b = bk.DrGhmcDiag(built, 3, [0.8, 0.4, 0.2], [2, 4, 8], 0.5, init=init, seed=17)
    assert "bk_user_drghmc" in a.compile_log and b.compile_log == ""
    da, la = a.sample_n(20)
    db, lb = b.sample_n(20)
    assert torch.equal(a.last_accept, b.last_accept) and torch.equal(a.last_n_uniform, b.last_n_uniform)
    assert 0 < float(a.last_accept.float().mean()) < 1
    np.testing.assert_allclose(np_(da), np_(db), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(la), np_(lb), rtol=1e-12, atol=1e-12)


# ---- 5. shards and the host surface, fp32 -------------------------------------------------------------------------
def test_shard_invariance_and_host_draws(bk, fused):
    D = 6
    dm = bk.CudaModel(BANANA, D, params=[0.5])
    init = np.random.default_rng(2).normal(size=(64, D))

    def make(**kw):
        return bk.DrGhmcDiag(dm, 3, [0.6, 0.3, 0.15], [2, 4, 8], 0.5, seed=9, **kw)

    full = make(init=init)
    fd, fl = full.sample_n(10)
    part = make(init=init[40:64], chain_offset=40)
    pd, pl = part.sample_n(10)
    assert torch.equal(fd[:, 40:64], pd) and torch.equal(fl[:, 40:64], pl)
    assert torch.equal(full.last_n_uniform[:, 40:64], part.last_n_uniform)
    assert torch.equal(full.rho[40:64], part.rho)

    ref = make(chains=256)
    rd, rl = ref.sample_n(5)
    for chunk in (None, 100, [100, 100, 56]):
        h = make(chains=256)
        hd, hl = h.sample_host_n(5, chunk_chains=chunk)
        assert torch.equal(rd.cpu(), hd) and torch.equal(rl.cpu(), hl)
        assert torch.equal(ref.last_accept, h.last_accept)
        assert torch.equal(ref.last_n_uniform[-1], h.last_n_uniform[-1])   # one launch per draw: the last draw's
        h1 = make(chains=256)
        d1, l1 = h1.sample_host(chunk_chains=chunk)
        assert torch.equal(rd[0].cpu(), d1) and torch.equal(rl[0].cpu(), l1)
        assert torch.equal(ref.last_n_uniform[0], h1.last_n_uniform[0])

    s = make(chains=256)
    d1, _ = s.sample_n(9, moments=True)
    d2, _ = s.sample_n(7, moments=True)
    np.testing.assert_allclose(np_(s.running_rhat()), np_(bk.rhat(torch.cat([d1, d2]), draws_first=True)), rtol=1e-4)


# ---- 6. statistics, fp32 ------------------------------------------------------------------------------------------
def test_banana_moments(bk, fused):
    """x1 has mean b and variance 1 + 2 b^2, every other coordinate is N(0, 1); within 4 MCSE."""
    b, D = 0.5, 8
    dm = bk.CudaModel(BANANA, D, params=[b])
    s = bk.DrGhmcDiag(dm, 3, [0.4, 0.2, 0.1], [4, 8, 16], 0.5, chains=2048, seed=3)
    assert "bk_user_drghmc" in s.compile_log
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


# ---- 7. engine choice and surface ---------------------------------------------------------------------------------
def test_engine_choice_and_surface(bk, fused):
    lib = bk._lib.lib()
    for D, want_fused in ((32, True), (33, False)):
        dm = bk.CudaModel(BANANA, D, params=[0.5])
        model_log = dm.compile_log
        s = bk.DrGhmcDiag(dm, 2, [0.3, 0.15], [2, 4], 0.5, chains=128, seed=1)
        assert dm.compile_log == model_log
        assert "bk_user_drghmc" not in model_log
        if want_fused:
            assert "Function properties for bk_user_drghmc" in s.compile_log
            with pytest.raises(NotImplementedError):
                s.sample_n(2, layout="series")
        else:
            assert s.compile_log == ""
        s.sample_n(1)
        n0 = lib.bk_launch_count()
        s.sample_n(3, keep_draws=False)
        launches = lib.bk_launch_count() - n0
        assert (launches == 1) if want_fused else (launches > 3), launches


def test_compile_error_raises_value_error(bk):
    # compiles as a model; its DrGHMC program (-DBK_DRGHMC=1) does not
    src = "#ifdef BK_DRGHMC\n#error no DrGHMC for this model\n#endif\n" + BANANA
    dm = bk.CudaModel(src, 3, params=[0.5])
    with pytest.raises(ValueError, match="no DrGHMC for this model"):
        bk.DrGhmcDiag(dm, 2, [0.3, 0.15], [2, 4], 0.5, chains=4)
