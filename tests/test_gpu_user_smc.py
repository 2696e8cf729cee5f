"""CudaPriorLikModel: user-written log prior / log likelihood pairs compiled at run time, and TemperedLikelihoodSMC on
them (one thread per particle, runtime-compiled move + weight kernel).  Each model is written twice, in CUDA for the
device and in NumPy for the oracle (oracle.samplers.smc_tempered takes any model with log_prior[_gradient] /
log_likelihood[_gradient])."""
import math

import numpy as np
import pytest
import torch

from _dev import device_model, np_, smc_kernel
from _user_cuda import GPL, MIX_MU, MIX_S, MIX_TAU, MIXTURE_MODEL, Mixture, binom, gpl, run_fake, user_twin
from conftest import GOLDEN, golden
from oracle import samplers as osm
from oracle import models as om

pytestmark = pytest.mark.gpu


def oracle_kernel(kind, scale, steps=5):
    return {"rw": ("rw", scale), "mala": ("mala", scale), "hmc": ("hmc", scale, steps)}[kind]


def device_kernel(bk, kind, scale, steps=5):
    return {"rw": lambda: bk.metropolis_kernel(scale), "mala": lambda: bk.mala_kernel(scale),
            "hmc": lambda: bk.hmc_kernel(scale, steps)}[kind]()


# ---- 1. protocol ---------------------------------------------------------------------------------------------------
def test_protocol_matches_the_oracle(bk):
    rng = np.random.default_rng(0)
    D = 7
    m0, p0, mu, pl = rng.normal(size=D), rng.uniform(0.5, 2, D), rng.normal(size=D), rng.uniform(1, 4, D)
    th = rng.normal(size=(33, D))
    ob = om.Binomial(2.0, 3.0, 7, 20)
    tb = rng.normal(size=(33, 1)) * 2
    for dm, nm, x in ((gpl(bk, m0, p0, mu, pl), om.GaussPriorLik(m0, p0, mu, pl), th),
                      (binom(bk, 2.0, 3.0, 7, 20), ob, tb)):
        np.testing.assert_allclose(np_(dm.log_prior(x)), [nm.log_prior(t) for t in x], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(np_(dm.log_likelihood(x)), [nm.log_likelihood(t) for t in x], rtol=1e-12, atol=1e-12)
        lp, g = dm.log_density_gradient(x)
        want = [nm.log_density_gradient(t) if hasattr(nm, "log_density_gradient")
                else (nm.log_density(t), nm.log_likelihood_gradient(t) + nm.log_prior_gradient(t)) for t in x]
        np.testing.assert_allclose(np_(lp), [w[0] for w in want], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(np_(g), np.stack([w[1] for w in want]), rtol=1e-12, atol=1e-12)
        assert isinstance(dm.log_prior(x[0]), float)
    # the built-in GaussPriorLik evaluates the same functions
    built = bk.GaussPriorLik(m0, p0, mu, pl, dtype=torch.float64)
    np.testing.assert_allclose(np_(gpl(bk, m0, p0, mu, pl).log_density(th)), np_(built.log_density(th)), rtol=1e-12)


def test_derived_density_runs_hmc_like_the_builtin(bk):
    """HMCDiag on the restated GaussPriorLik == on the built-in plugin (fp64, Philox): the derived
    log_density_gradient = ll + prior, gll + gpr is the posterior's."""
    rng = np.random.default_rng(1)
    D = 6
    m0, p0, mu, pl = np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D)
    init = rng.normal(size=(64, D))
    a = bk.HMCDiag(gpl(bk, m0, p0, mu, pl), 0.2, 5, init=init, seed=3)
    b = bk.HMCDiag(bk.GaussPriorLik(m0, p0, mu, pl, dtype=torch.float64), 0.2, 5, init=init, seed=3)
    da, la = a.sample_n(20)
    db, lb = b.sample_n(20)
    assert torch.equal(a.last_accept, b.last_accept)
    assert 0 < float(a.last_accept.float().mean()) < 1
    np.testing.assert_allclose(np_(da), np_(db), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(la), np_(lb), rtol=1e-12, atol=1e-12)


# ---- 2. the reference's own runs -------------------------------------------------------------------------------
def _smc_names():
    import glob
    import os
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "smc_*.npz")))


@pytest.mark.parametrize("name", _smc_names())
def test_smc_golden_through_the_user_model(bk, name):
    """The recorded legacy-RNG streams of the reference (tests/golden/smc_*): bit-exact multinomial indices at every
    temperature and the final particles within 1e-10, with the restated model in place of the built-in."""
    z = golden(name)
    model = user_twin(bk, z)
    M, T = z["thetas0"].shape[0], int(z["T"])
    smc = bk.TemperedLikelihoodSMC(model, M, T, z["thetas0"], smc_kernel(bk, z))
    for n in range(1, T + 1):
        smc.transition(n, normals=z["normals"][n - 1], acc_uniforms=z["acc_uniforms"][n - 1],
                       res_uniforms=z["res_uniforms"][n - 1])
        assert np.array_equal(np_(smc.last_indices), z["indices"][n - 1]), f"indices differ at n={n}"
    np.testing.assert_allclose(np_(smc.thetas), z["thetas_final"], rtol=1e-10, atol=1e-10)


# ---- 3. a model with no built-in counterpart ---------------------------------------------------------------------
@pytest.mark.parametrize("kind,scale", [("rw", 0.3), ("mala", 0.05), ("hmc", 0.1)])
@pytest.mark.parametrize("mode", ["systematic", "multinomial"])
def test_mixture_vs_oracle(bk, kind, scale, mode):
    rng = np.random.default_rng(21)
    nm = Mixture(MIX_MU, MIX_S, MIX_TAU)
    D, M, T = 4, 203, 6
    th0 = rng.normal(size=(M, D)) * MIX_TAU
    zs, au, ru = rng.standard_normal((T, M, D)), rng.random((T, M)), rng.random((T, M))
    oth, oidx = osm.smc_tempered(nm, th0, zs, au, ru, scale, T, resample=mode, kernel=oracle_kernel(kind, scale))
    dm = bk.CudaPriorLikModel(MIXTURE_MODEL, D, params=nm.params(), dtype=torch.float64)
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, device_kernel(bk, kind, scale), resample=mode)
    acc = []
    for n in range(1, T + 1):
        r = ru[n - 1, :1] if mode == "systematic" else ru[n - 1]
        smc.transition(n, normals=zs[n - 1], acc_uniforms=au[n - 1], res_uniforms=r)
        acc.append(float(smc.last_accept.float().mean()))
        assert np.array_equal(np_(smc.last_indices), oidx[n - 1]), f"indices differ at n={n}"
    assert 0 < np.mean(acc) < 1
    tol = 1e-12 if mode == "systematic" else 1e-10
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=tol, atol=tol)


def _mixture_stats(bk, kind, seed, M=1 << 16, T=40):
    nm = Mixture(MIX_MU, MIX_S, MIX_TAU)
    dm = bk.CudaPriorLikModel(MIXTURE_MODEL, 4, params=nm.params())
    th0 = torch.randn(M, 4, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)) * MIX_TAU
    scale = {"rw": 0.3, "mala": 0.05, "hmc": 0.1}[kind]
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, device_kernel(bk, kind, scale), resample="systematic", seed=seed)
    smc.run()
    th = np_(smc.thetas).astype(np.float64)
    up = th @ MIX_MU > 0
    return up.mean(), th[up].mean(0), th[~up].mean(0)


@pytest.mark.parametrize("kind", ["rw", "mala", "hmc"])
def test_mixture_posterior_fp32(bk, kind):
    """fp32 Philox, M = 2^16: by symmetry half of the particles sit in each mode, and each mode's mean is the conjugate
    mean mu tau^2 / (tau^2 + s^2) (the modes are ~6 posterior sd from the plane between them).  The tolerances are
    four times the spread of the replicate seeds run here (and at least the Monte-Carlo error of 2^16 particles)."""
    want = MIX_MU * MIX_TAU ** 2 / (MIX_TAU ** 2 + MIX_S ** 2)
    reps = [_mixture_stats(bk, kind, seed) for seed in (1, 2, 3, 4)]
    frac = np.array([r[0] for r in reps])
    mean_up = np.array([r[1] for r in reps])
    mean_dn = np.array([r[2] for r in reps])
    tol_f = max(4 * frac.std(ddof=1), 4 * math.sqrt(0.25 / (1 << 16)))
    tol_m = max(4 * max(mean_up.std(0, ddof=1).max(), mean_dn.std(0, ddof=1).max()), 0.02)
    assert tol_f < 0.05 and tol_m < 0.1, (frac, mean_up, mean_dn)      # the replicate spread itself is small
    assert abs(frac.mean() - 0.5) < tol_f, frac
    np.testing.assert_allclose(mean_up.mean(0), want, atol=tol_m)
    np.testing.assert_allclose(mean_dn.mean(0), -want, atol=tol_m)


# ---- 4. same RNG as the built-in ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,scale", [("rw", 0.25), ("mala", 0.05), ("hmc", 0.1)])
def test_same_streams_as_the_builtin(bk, kind, scale):
    """fp64 Philox: the restated GaussPriorLik consumes the built-in's Philox words (normals of element blocks,
    accept uniform of block ceil(D / 4)): identical indices and accept flags, particles within 1e-12."""
    rng = np.random.default_rng(4)
    D, M, T = 6, 1000, 4
    m0, p0, mu, pl = np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D)
    th0 = rng.normal(size=(M, D))
    runs = []
    for model in (gpl(bk, m0, p0, mu, pl), bk.GaussPriorLik(m0, p0, mu, pl, dtype=torch.float64)):
        smc = bk.TemperedLikelihoodSMC(model, M, T, th0, device_kernel(bk, kind, scale), resample="systematic", seed=8)
        idx, acc = [], []
        for n in range(1, T + 1):
            smc.transition(n)
            idx.append(np_(smc.last_indices).copy())
            acc.append(np_(smc.last_accept).copy())
        runs.append((np.stack(idx), np.stack(acc), np_(smc.thetas)))
    (iu, au, tu), (ib, ab, tb) = runs
    assert np.array_equal(iu, ib)
    assert np.array_equal(au, ab) and 0 < au.mean() < 1
    np.testing.assert_allclose(tu, tb, rtol=1e-12, atol=1e-12)


# ---- 5. sharding -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [1, 2, 3, 5])
@pytest.mark.parametrize("mode", ["systematic", "multinomial"])
def test_sharded_user_smc_equals_oracle(bk, world, mode):
    rng = np.random.default_rng(5)
    nm = Mixture(MIX_MU, MIX_S, MIX_TAU)
    D, M, T, scale = 4, 211, 5, 0.3           # 211 is prime: ragged shards for every world > 1
    th0 = rng.normal(size=(M, D)) * MIX_TAU
    zs, au, ru = rng.standard_normal((T, M, D)), rng.random((T, M)), rng.random((T, M))
    oth, oidx = osm.smc_tempered(nm, th0, zs, au, ru, scale, T, resample=mode)
    dm = bk.CudaPriorLikModel(MIXTURE_MODEL, D, params=nm.params(), dtype=torch.float64)

    def make(group):
        return bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.metropolis_kernel(scale), resample=mode, group=group)

    def streams(n, lo, hi, s):
        r = ru[n - 1, :1] if mode == "systematic" else ru[n - 1, lo:hi]
        return zs[n - 1, lo:hi], au[n - 1, lo:hi], r

    idx, th, ranks = run_fake(bk, world, make, T, streams)
    assert np.array_equal(idx, oidx), f"indices differ (world={world}, {mode})"
    np.testing.assert_allclose(th, oth, rtol=1e-12, atol=1e-12)
    for s in ranks[1:]:
        assert s.weight_ess == ranks[0].weight_ess


@pytest.mark.parametrize("kind", ["rw", "mala", "hmc"])
def test_sharded_user_smc_philox_invariant(bk, kind):
    """fp32 device Philox: world 1, 3 and 8 give bit-identical particles and indices, equal to one unsharded run()
    -- the peer row reads, the (ll, prior) carry and the mailbox max of the runtime-compiled kernel."""
    M, T, D = 20011, 6, 8
    g = torch.Generator(device="cuda").manual_seed(1)
    mu = torch.randn(D, device="cuda", generator=g)
    th0 = torch.randn(M, D, device="cuda", generator=g)
    dm = gpl(bk, np.zeros(D), np.ones(D), mu.cpu().numpy(), 4 * np.ones(D), dtype=torch.float32)
    kern = device_kernel(bk, kind, {"rw": 0.2, "mala": 0.05, "hmc": 0.1}[kind])

    def make(group):
        return bk.TemperedLikelihoodSMC(dm, M, T, th0, kern, resample="systematic", seed=7, group=group)

    none = lambda n, lo, hi, s: (None, None, None)
    idx1, th1, _ = run_fake(bk, 1, make, T, none)
    for world in (3, 8):
        idxg, thg, _ = run_fake(bk, world, make, T, none)
        assert np.array_equal(idx1, idxg), world
        assert np.array_equal(th1, thg), world
    single = bk.TemperedLikelihoodSMC(dm, M, T, th0, kern, resample="systematic", seed=7)
    single.run()
    assert np.array_equal(np_(single.thetas), th1)


# ---- 6. adaptive resampling ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("thr", [0.5, 1.0])
def test_user_smc_adaptive_vs_oracle(bk, thr):
    rng = np.random.default_rng(11)
    nm = Mixture(MIX_MU, MIX_S, MIX_TAU)
    D, M, T, scale = 4, 300, 12, 0.3
    th0 = rng.normal(size=(M, D)) * MIX_TAU
    zs, au, ru = rng.standard_normal((T, M, D)), rng.random((T, M)), rng.random((T, M))
    oth, ologw, oflags = osm.smc_tempered_adaptive(nm, th0, zs, au, ru, scale, T, thr)
    dm = bk.CudaPriorLikModel(MIXTURE_MODEL, D, params=nm.params(), dtype=torch.float64)
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.metropolis_kernel(scale), resample="systematic",
                                   ess_threshold=thr)
    for n in range(1, T + 1):
        smc.transition(n, normals=zs[n - 1], acc_uniforms=au[n - 1], res_uniforms=ru[n - 1, :1])
    assert smc.resampled == list(oflags)
    if thr < 1.0:
        assert 0 < sum(oflags) < T
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(smc.log_weights), ologw, rtol=1e-10, atol=1e-12)


# ---- 7. surface and errors ----------------------------------------------------------------------------------------
def test_surface_and_errors(bk):
    plain = bk.CudaModel("""
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    g[0] = -x[0]; g[1] = -x[1];
    return bk_real(-0.5) * (x[0] * x[0] + x[1] * x[1]);
}""", 2)
    with pytest.raises(TypeError, match="log_prior/log_likelihood"):
        bk.TemperedLikelihoodSMC(plain, 64, 3, np.zeros((64, 2)), bk.metropolis_kernel(0.3))
    with pytest.raises(ValueError, match="dims"):
        bk.CudaPriorLikModel(GPL, 257, params=np.ones(4 * 257))
    bad = GPL.replace("return quad(x, g, p, p + BK_DIMS);", "return quad(x, g, p, p + BK_DIMS)")
    with pytest.raises(ValueError, match=r"model.cu\(\d+\): error"):
        bk.CudaPriorLikModel(bad, 3, params=np.ones(12))
    with pytest.raises(ValueError, match="log_likelihood_gradient"):
        bk.CudaPriorLikModel(GPL[:GPL.index("__device__ bk_real log_likelihood_gradient")], 3, params=np.ones(12))
    # run(), then transition() steps, then .thetas; last_accept [M_local] in {0, 1}
    nm = Mixture(MIX_MU, MIX_S, MIX_TAU)
    dm = bk.CudaPriorLikModel(MIXTURE_MODEL, 4, params=nm.params())
    assert "bk_user_smc_hmc" in dm.compile_log
    M, T = 1000, 8
    smc = bk.TemperedLikelihoodSMC(dm, M, T, lambda m: np.full(4, 0.1 * (m % 7)), bk.hmc_kernel(0.1, 3),
                                   resample="systematic", seed=2)
    smc.run_steps(1, 5)
    for n in range(6, T + 1):
        smc.transition(n)
    th = smc.thetas
    assert th.shape == (M, 4) and torch.isfinite(th).all()
    acc = smc.last_accept
    assert acc.shape == (M,) and set(np_(acc).tolist()) <= {0, 1}
    assert len(smc.weight_ess) == T
    full = bk.TemperedLikelihoodSMC(dm, M, T, np.zeros((M, 4)), bk.mala_kernel(0.05), resample="multinomial", seed=2)
    full.run()
    assert full.thetas.shape == (M, 4) and torch.isfinite(full.thetas).all()
