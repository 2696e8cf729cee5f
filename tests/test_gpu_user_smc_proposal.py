"""TemperedLikelihoodSMC with a user-written CudaProposal as the move (proposal_kernel): one Metropolis(-Hastings) step
of the proposal on the tempered density, compiled together with a CudaPriorLikModel into one kernel
(bk_user_smc_mhp).  Models and proposals are written in CUDA for the device and in NumPy for the restatement in
tests/_smc_proposal_oracle.py; most of them, shared with test_gpu_user_smc.py and test_gpu_user_proposal.py, are
in tests/_user_cuda.py."""
import math

import numpy as np
import pytest
import torch

import _smc_proposal_oracle as sop
from _dev import np_
from _user_cuda import (GAMMA_POIS, GPL, INDEP, LOGNORMAL, MIX_MU, MIX_S, MIX_TAU, MIXTURE_MODEL, MIXTURE_WALK, RSCAN,
                        RW, GammaPois, Mixture, binom, gpl, np_indep, np_lognormal, np_mixture_walk, np_rscan,
                        philox_streams, run_fake, user_twin)
from conftest import golden

pytestmark = pytest.mark.gpu


def walk(bk, s, D, dtype, transition=False):
    return bk.CudaProposal(RW, D, params=[s], transition=transition, dtype=dtype)


def _gpl_model(bk, D, dtype, seed=0):
    if D == 1:
        return binom(bk, 2.0, 3.0, 7, 20, dtype=dtype)
    rng = np.random.default_rng(seed + D)
    return gpl(bk, np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D), dtype=dtype)


def _drive(smc, T, streams=None, run=False):
    """transition() steps (streams(n) -> (normals, acc_uniforms, res_uniforms)) or one run(); returns
    (indices [T, M], accept [T, M] (run: the last step only), particles)."""
    if run:
        smc.run()
        return np_(smc.last_indices)[None], np_(smc.last_accept)[None], smc.thetas.clone()
    idx, acc = [], []
    for n in range(1, T + 1):
        z, au, ru = streams(n) if streams else (None, None, None)
        smc.transition(n, normals=z, acc_uniforms=au, res_uniforms=ru)
        idx.append(np_(smc.last_indices).copy())
        acc.append(np_(smc.last_accept).copy())
    return np.stack(idx), np.stack(acc), smc.thetas.clone()


# ---- 1. the random walk restated is metropolis_kernel ---------------------------------------------------------------
@pytest.mark.parametrize("rng_mode,drive", [("philox", "transition"), ("philox", "run"), ("injected", "transition")])
@pytest.mark.parametrize("mode", ["systematic", "multinomial"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("D", [1, 2, 5, 17, 50])
def test_walk_restated_equals_metropolis_kernel(bk, D, dtype, rng_mode, drive, mode):
    """Same streams and the same arithmetic as bk_user_smc_rw: indices, accept flags and particles equal bit for bit,
    in fp32 too (NVRTC contracts theta + s * z into one FMA in both kernels).  run() draws from Philox; injected
    streams go through transition()."""
    M, T, seed = 301, 4, 5
    s = 0.8 if D == 1 else min(0.3, 1.0 / math.sqrt(D))
    model = _gpl_model(bk, D, dtype)
    th0 = np.random.default_rng(D).normal(size=(M, D)) * 0.5
    g = np.random.default_rng(100 + D)
    zs, au, ru = g.standard_normal((T, M, D)), g.random((T, M)), g.random((T, M))

    def streams(n):
        if rng_mode == "philox":
            return None, None, None
        return zs[n - 1], au[n - 1], (ru[n - 1, :1] if mode == "systematic" else ru[n - 1])

    runs = []
    for kern in (bk.proposal_kernel(walk(bk, s, D, dtype)), bk.metropolis_kernel(s)):
        smc = bk.TemperedLikelihoodSMC(model, M, T, th0, kern, resample=mode, seed=seed)
        runs.append(_drive(smc, T, streams, run=drive == "run"))
    (ip, ap, tp), (ir, ar, tr) = runs
    assert np.array_equal(ip, ir)
    assert np.array_equal(ap, ar) and 0 < ap.mean() < 1
    assert torch.equal(tp, tr)


# ---- 2. the reference's own runs --------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["smc_gauss_d5", "smc_gauss_d50", "smc_binom"])
def test_rw_goldens_through_the_restated_walk(bk, name):
    """The reference's recorded streams (tests/golden/smc_*) through the proposal move: bit-exact multinomial indices
    at every temperature and the final particles within 1e-10."""
    z = golden(name)
    model = user_twin(bk, z)
    M, T, D = z["thetas0"].shape[0], int(z["T"]), z["thetas0"].shape[1]
    smc = bk.TemperedLikelihoodSMC(model, M, T, z["thetas0"],
                                   bk.proposal_kernel(walk(bk, float(z["scale"]), D, torch.float64)))
    for n in range(1, T + 1):
        smc.transition(n, normals=z["normals"][n - 1], acc_uniforms=z["acc_uniforms"][n - 1],
                       res_uniforms=z["res_uniforms"][n - 1])
        assert np.array_equal(np_(smc.last_indices), z["indices"][n - 1]), f"indices differ at n={n}"
    np.testing.assert_allclose(np_(smc.thetas), z["thetas_final"], rtol=1e-10, atol=1e-10)


# ---- 3. Hastings and uniform-consuming proposals against the restatement ---------------------------------------------
GP = GammaPois(2.0, 1.0, 4.0, [3.0, 5.0, 8.0, 2.0])
GP_MEAN = (GP.a + GP.S) / (GP.b + GP.n)


def _case(bk, which, dtype=torch.float64):
    """(device model, NumPy model, device proposal, propose, transition, initial particles [M, D] generator)."""
    if which in ("lognormal", "indep"):
        dm = bk.CudaPriorLikModel(GAMMA_POIS, 4, params=GP.params(), dtype=dtype)
        init = lambda rng, M: rng.gamma(GP.a, 1.0 / GP.b, size=(M, 4))
        if which == "lognormal":
            prop = bk.CudaProposal(LOGNORMAL, 4, params=[0.4], dtype=dtype)
            p, t = np_lognormal(0.4)
        else:
            m, s = GP_MEAN, np.full(4, 0.8)
            prop = bk.CudaProposal(INDEP, 4, params=np.concatenate([m, s]), dtype=dtype)
            p, t = np_indep(m, s)
        return dm, GP, prop, p, t, init
    nm = Mixture(MIX_MU, MIX_S, MIX_TAU)
    dm = bk.CudaPriorLikModel(MIXTURE_MODEL, 4, params=nm.params(), dtype=dtype)
    init = lambda rng, M: rng.normal(size=(M, 4)) * MIX_TAU
    if which == "rscan":
        prop = bk.CudaProposal(RSCAN, 4, params=[0.8], normals=1, uniforms=1, dtype=dtype)
        p, t = np_rscan(0.8)
        return dm, nm, prop, p, t, init
    prop = bk.CudaProposal(MIXTURE_WALK, 4, params=[0.3, 1.2, 0.6], normals=8, uniforms=2, transition=False,
                           dtype=dtype)
    return dm, nm, prop, np_mixture_walk(0.3, 1.2, 0.6), None, init


def _streams(rng, T, M, prop):
    zs = rng.standard_normal((T, M, prop.normals))
    au = rng.random((T, M, 1 + prop.uniforms))
    return zs, au, rng.random((T, M))


@pytest.mark.parametrize("mode", ["systematic", "multinomial"])
@pytest.mark.parametrize("which", ["lognormal", "indep", "rscan", "mixprop"])
def test_proposals_vs_restatement(bk, which, mode):
    rng = np.random.default_rng(31)
    dm, nm, prop, p, t, init = _case(bk, which)
    M, T = 203, 6
    th0 = init(rng, M)
    zs, au, ru = _streams(rng, T, M, prop)
    oth, oidx, oacc = sop.smc_tempered(nm, th0, zs, au, ru, T, p, t, resample=mode)
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.proposal_kernel(prop), resample=mode)
    for n in range(1, T + 1):
        r = ru[n - 1, :1] if mode == "systematic" else ru[n - 1]
        smc.transition(n, normals=zs[n - 1], acc_uniforms=au[n - 1], res_uniforms=r)
        assert np.array_equal(np_(smc.last_accept).astype(bool), oacc[n - 1]), f"accept flags differ at n={n}"
        assert np.array_equal(np_(smc.last_indices), oidx[n - 1]), f"indices differ at n={n}"
    assert 0 < oacc.mean() < 1
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=1e-10, atol=1e-10)


# ---- 4. Philox equals the injected reconstruction ---------------------------------------------------------------------
@pytest.mark.parametrize("which", ["lognormal", "mixprop"])
def test_philox_equals_injected_reconstruction(bk, which):
    """fp64, three ranks (chain_offset = lo(rank) > 0 on ranks 1 and 2), temperatures n = 1..4: the streams rebuilt
    outside the library (bk_init_normal blocks without the accept block, the restated uniforms) reproduce the Philox
    run exactly."""
    dm, _, prop, _, _, init = _case(bk, which)
    M, T, seed, world = 97, 4, 123, 3
    th0 = init(np.random.default_rng(2), M)

    def make(group):
        return bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.proposal_kernel(prop), resample="systematic", seed=seed,
                                        group=group)

    rs = np.random.default_rng(3).random((T, 1))

    def rebuilt(n, lo, hi, s):
        Z, U = philox_streams(bk, seed, lo, hi - lo, 4, prop.normals, prop.uniforms, 1, n)
        return Z[0], U[0], rs[n - 1]

    idx_p, th_p, ranks = run_fake(bk, world, make, T, lambda n, lo, hi, s: (None, None, rs[n - 1]))
    idx_i, th_i, _ = run_fake(bk, world, make, T, rebuilt)
    assert np.array_equal(idx_p, idx_i)
    assert np.array_equal(th_p, th_i)
    assert 0 < float(ranks[0].last_accept.float().mean()) < 1


# ---- 5. sharding ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [1, 2, 3, 5])
@pytest.mark.parametrize("mode", ["systematic", "multinomial"])
def test_sharded_equals_restatement(bk, world, mode):
    rng = np.random.default_rng(5)
    dm, nm, prop, p, t, init = _case(bk, "rscan")
    M, T = 211, 5                              # 211 is prime: ragged shards for every world > 1
    th0 = init(rng, M)
    zs, au, ru = _streams(rng, T, M, prop)
    oth, oidx, _ = sop.smc_tempered(nm, th0, zs, au, ru, T, p, t, resample=mode)

    def make(group):
        return bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.proposal_kernel(prop), resample=mode, group=group)

    def streams(n, lo, hi, s):
        r = ru[n - 1, :1] if mode == "systematic" else ru[n - 1, lo:hi]
        return zs[n - 1, lo:hi], au[n - 1, lo:hi], r

    idx, th, _ = run_fake(bk, world, make, T, streams)
    assert np.array_equal(idx, oidx), f"indices differ (world={world}, {mode})"
    np.testing.assert_allclose(th, oth, rtol=1e-10, atol=1e-10)


def test_sharded_philox_invariant_fp32(bk):
    """fp32 device Philox: world 1, 3 and 8 give bit-identical particles and indices, equal to one unsharded run()."""
    M, T, D = 20011, 6, 8
    g = torch.Generator(device="cuda").manual_seed(1)
    mu = torch.randn(D, device="cuda", generator=g)
    th0 = torch.randn(M, D, device="cuda", generator=g)
    dm = gpl(bk, np.zeros(D), np.ones(D), mu.cpu().numpy(), 4 * np.ones(D), dtype=torch.float32)
    prop = bk.CudaProposal(MIXTURE_WALK, D, params=[0.15, 0.4, 0.6], normals=2 * D, uniforms=2, transition=False)
    kern = bk.proposal_kernel(prop)

    def make(group):
        return bk.TemperedLikelihoodSMC(dm, M, T, th0, kern, resample="systematic", seed=7, group=group)

    none = lambda n, lo, hi, s: (None, None, None)
    idx1, th1, r1 = run_fake(bk, 1, make, T, none)
    assert 0 < float(r1[0].last_accept.float().mean()) < 1
    for world in (3, 8):
        idxg, thg, _ = run_fake(bk, world, make, T, none)
        assert np.array_equal(idx1, idxg), world
        assert np.array_equal(th1, thg), world
    single = bk.TemperedLikelihoodSMC(dm, M, T, th0, kern, resample="systematic", seed=7)
    single.run()
    assert np.array_equal(np_(single.thetas), th1)


@pytest.mark.parametrize("thr", [0.5, 1.0])
def test_adaptive_vs_restatement(bk, thr):
    rng = np.random.default_rng(11)
    dm, nm, prop, p, t, init = _case(bk, "lognormal")
    M, T = 300, 12
    th0 = init(rng, M)
    zs, au, ru = _streams(rng, T, M, prop)
    oth, ologw, oflags = sop.smc_tempered_adaptive(nm, th0, zs, au, ru, T, thr, p, t)
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.proposal_kernel(prop), resample="systematic", ess_threshold=thr)
    for n in range(1, T + 1):
        smc.transition(n, normals=zs[n - 1], acc_uniforms=au[n - 1], res_uniforms=ru[n - 1, :1])
    assert smc.resampled == list(oflags)
    if thr < 1.0:
        assert 0 < sum(oflags) < T
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(np_(smc.log_weights), ologw, rtol=1e-10, atol=1e-12)


# ---- 6. statistics ----------------------------------------------------------------------------------------------------
def _gamma_stats(bk, transition, seed, M=1 << 16, T=40):
    dm = bk.CudaPriorLikModel(GAMMA_POIS, 4, params=GP.params())
    prop = bk.CudaProposal(LOGNORMAL, 4, params=[0.4], transition=transition)
    th0 = np.random.default_rng(seed).gamma(GP.a, 1.0 / GP.b, size=(M, 4))
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.proposal_kernel(prop), resample="systematic", seed=seed)
    smc.run()
    th = np_(smc.thetas).astype(np.float64)
    return th.mean(0), th.var(0)


def test_gamma_poisson_posterior_fp32(bk):
    """fp32 Philox, M = 2^16, the log-normal walk with its Hastings term: the posterior is Gamma(a + S, b + n), mean
    (a + S) / (b + n), variance (a + S) / (b + n)^2.  Tolerances: four times the spread of the replicate seeds (and at
    least the Monte-Carlo error of 2^16 particles).  Without the Hastings term the same walk leaves the tempered
    posteriors invariant only up to the Jacobian: its mean must miss by far more than that tolerance."""
    want_m, want_v = GP_MEAN, (GP.a + GP.S) / (GP.b + GP.n) ** 2
    reps = [_gamma_stats(bk, True, seed) for seed in (1, 2, 3, 4)]
    mean, var = np.array([r[0] for r in reps]), np.array([r[1] for r in reps])
    tol_m = max(4 * mean.std(0, ddof=1).max(), 4 * math.sqrt(want_v.max() / (1 << 16)))
    tol_v = max(4 * var.std(0, ddof=1).max(), 4 * math.sqrt(2 / (1 << 16)) * want_v.max())
    assert tol_m < 0.05 and tol_v < 0.05, (mean, var)          # the replicate spread itself is small
    np.testing.assert_allclose(mean.mean(0), want_m, atol=tol_m)
    np.testing.assert_allclose(var.mean(0), want_v, atol=tol_v)
    wrong = np.array([_gamma_stats(bk, False, seed)[0] for seed in (1, 2)]).mean(0)
    assert np.abs(wrong - want_m).max() > 4 * tol_m, (wrong, want_m, tol_m)


# ---- 7. errors ----------------------------------------------------------------------------------------------------------
def test_errors(bk):
    D = 3
    prop = walk(bk, 0.3, D, torch.float64)
    th0 = np.zeros((64, D))
    for built in (bk.GaussPriorLik(np.zeros(D), np.ones(D), np.zeros(D), np.ones(D), dtype=torch.float64),
                  bk.Binomial(2.0, 3.0, 7, 20, dtype=torch.float64)):
        p = prop if built.dims() == D else walk(bk, 0.3, 1, torch.float64)
        with pytest.raises(NotImplementedError, match="CudaPriorLikModel"):
            bk.TemperedLikelihoodSMC(built, 64, 3, np.zeros((64, built.dims())), bk.proposal_kernel(p))
    plain = bk.CudaModel("""
__device__ bk_real log_density_gradient(const bk_real* x, bk_real* g, const bk_real* p) {
    bk_real s = 0; for (int e = 0; e < BK_DIMS; ++e) { s += x[e] * x[e]; g[e] = -x[e]; } return bk_real(-0.5) * s;
}""", D, dtype=torch.float64)
    with pytest.raises(TypeError, match="log_prior/log_likelihood"):
        bk.TemperedLikelihoodSMC(plain, 64, 3, th0, bk.proposal_kernel(prop))
    model = _gpl_model(bk, D, torch.float64)
    with pytest.raises(ValueError, match="does not match the model"):
        bk.TemperedLikelihoodSMC(model, 64, 3, th0, bk.proposal_kernel(walk(bk, 0.3, D + 1, torch.float64)))
    with pytest.raises(ValueError, match="does not match the model"):
        bk.TemperedLikelihoodSMC(model, 64, 3, th0, bk.proposal_kernel(walk(bk, 0.3, D, torch.float32)))
    big = bk.CudaProposal(RW, D, params=[0.3], normals=513, dtype=torch.float64)
    with pytest.raises(ValueError, match="n_normals <= 512"):
        bk.TemperedLikelihoodSMC(model, 64, 3, th0, bk.proposal_kernel(big))
    uni = bk.CudaProposal(RSCAN, D, params=[0.8], normals=1, uniforms=1, dtype=torch.float64)
    smc = bk.TemperedLikelihoodSMC(model, 64, 3, th0, bk.proposal_kernel(uni))
    with pytest.raises(ValueError, match="acc_uniforms"):
        smc.transition(1, normals=np.zeros((64, 1)), acc_uniforms=np.full(64, 0.5), res_uniforms=np.full(64, 0.5))
    with pytest.raises(TypeError, match="CudaProposal"):
        bk.proposal_kernel(bk.GaussianRW(0.3))
    # the kernel keeps its proposal alive
    k = bk.proposal_kernel(walk(bk, 0.3, D, torch.float64))
    smc = bk.TemperedLikelihoodSMC(model, 64, 3, th0, k, resample="systematic", seed=1)
    smc.run()
    assert torch.isfinite(smc.thetas).all()


# ---- 8. what was compiled ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [1, 50, 256])
def test_compile_log_lists_the_kernel(bk, D):
    rng = np.random.default_rng(D)
    model = gpl(bk, np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D), dtype=torch.float32)
    th0 = np.zeros((128, D))
    for prop in (bk.CudaProposal(RW, D, params=[0.3], transition=True),
                 bk.CudaProposal(RW, D, params=[0.3], transition=False),
                 bk.CudaProposal(RSCAN, D, params=[0.8], normals=1, uniforms=1)):
        smc = bk.TemperedLikelihoodSMC(model, 128, 2, th0, bk.proposal_kernel(prop))
        assert "Function properties for bk_user_smc_mhp" in smc.compile_log
    if D <= 32:   # the fused MCMC program of a plain model with the same proposal holds no SMC kernel
        plain = bk.CudaModel(GPL.replace("log_prior_gradient", "lpg").replace(
            "log_likelihood_gradient", "log_density_gradient"), D, params=np.ones(4 * D))
        mh = bk.Metropolis(plain, bk.CudaProposal(RW, D, params=[0.3], transition=False), init=np.zeros((8, D)))
        assert "bk_user_mhp" in mh.compile_log and "bk_user_smc_mhp" not in mh.compile_log
