"""TemperedLikelihoodSMC(..., moves=k): k applications of the Markov kernel per particle and temperature, fused into
the move + weight kernel, against the fp64 oracle's composed kernel, the built-in plugins against their CUDA
restatements, sharded against single-rank runs, and statistically against the analytic posterior."""
import numpy as np
import pytest
import torch

import _smc_moves_oracle as mo
import _user_cuda as uc
from _dev import device_model, np_
from conftest import golden
from oracle import models as om
from oracle import samplers as osm

pytestmark = pytest.mark.gpu

KERNELS = {"rw": ("rw", 0.4), "mala": ("mala", 0.05), "hmc": ("hmc", 0.1, 3)}


def _dev_kernel(bk, kern):
    if kern[0] == "rw":
        return bk.metropolis_kernel(kern[1])
    if kern[0] == "mala":
        return bk.mala_kernel(kern[1])
    return bk.hmc_kernel(kern[1], kern[2])


def _models(bk, which, rng):
    if which == "binom":
        return bk.Binomial(2.0, 3.0, 7, 20, dtype=torch.float64), om.Binomial(2.0, 3.0, 7, 20), 1
    D = int(which[3:])
    mu = rng.normal(size=D)
    return (bk.GaussPriorLik(np.zeros(D), np.ones(D), mu, 4 * np.ones(D), dtype=torch.float64),
            om.GaussPriorLik(np.zeros(D), np.ones(D), mu, 4 * np.ones(D)), D)


def _streams(rng, T, M, k, D):
    return rng.standard_normal((T, M, k, D)), rng.random((T, M, k)), rng.random((T, M))


def _inject(smc, T, zs, au, ru, systematic, on_step=None):
    for n in range(1, T + 1):
        smc.transition(n, normals=zs[n - 1], acc_uniforms=au[n - 1], res_uniforms=ru[n - 1, :1] if systematic
                       else ru[n - 1])
        if on_step:
            on_step(n)


def test_explicit_one_move_is_the_default(bk):
    rng = np.random.default_rng(1)
    dm, _, D = _models(bk, "gpl5", rng)
    M, T = 500, 6
    th0 = rng.normal(size=(M, D))
    a = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.mala_kernel(0.05), resample="systematic", seed=4)
    b = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.mala_kernel(0.05), resample="systematic", seed=4, moves=1)
    a.run()
    b.run()
    assert torch.equal(a.thetas, b.thetas) and torch.equal(a.last_indices, b.last_indices)
    assert torch.equal(a.last_accept, b.last_accept)
    assert np.array_equal(a.weight_ess, b.weight_ess)


@pytest.mark.parametrize("resample", ["multinomial", "systematic"])
@pytest.mark.parametrize("kernel", ["rw", "mala", "hmc"])
@pytest.mark.parametrize("which", ["gpl5", "gpl50", "binom"])
@pytest.mark.parametrize("k", [2, 5])
def test_injected_fp64_matches_the_oracle(bk, which, kernel, resample, k):
    rng = np.random.default_rng(7)
    dm, nm, D = _models(bk, which, rng)
    M, T, kern = 48, 3, KERNELS[kernel]
    th0 = rng.normal(size=(M, D))
    zs, au, ru = _streams(rng, T, M, k, D)
    oth, oidx, oacc = mo.smc_tempered(nm, th0, zs, au, ru, T, kern, resample=resample)
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, _dev_kernel(bk, kern), resample=resample, moves=k)
    got_idx = []

    def step(n):   # last_accept: the accepted moves of each particle, in [0, k]
        got_idx.append(np_(smc.last_indices).copy())
        acc = np_(smc.last_accept)
        assert smc.last_accept.dtype == torch.int32 and acc.min() >= 0 and acc.max() <= k
        assert np.array_equal(acc, oacc[n - 1])
    _inject(smc, T, zs, au, ru, resample == "systematic", step)
    assert np.array_equal(np.stack(got_idx), oidx)
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("name", ["smc_gauss_d5", "smc_gauss_d50", "smc_binom"])
def test_zero_extra_normals_reproduce_the_goldens_on_device(bk, name):
    z = golden(name)
    k = 3
    T, M, D = z["normals"].shape
    zs = np.zeros((T, M, k, D))
    zs[:, :, 0] = z["normals"]
    au = np.full((T, M, k), 0.5)
    au[:, :, 0] = z["acc_uniforms"]
    smc = bk.TemperedLikelihoodSMC(device_model(bk, z), M, T, z["thetas0"], bk.metropolis_kernel(float(z["scale"])),
                                   moves=k)
    for n in range(1, T + 1):
        smc.transition(n, normals=zs[n - 1], acc_uniforms=au[n - 1], res_uniforms=z["res_uniforms"][n - 1])
        assert np.array_equal(np_(smc.last_indices), z["indices"][n - 1])
    np.testing.assert_allclose(np_(smc.thetas), z["thetas_final"], rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("kernel", ["rw", "mala", "hmc"])
@pytest.mark.parametrize("injected", [True, False])
def test_user_model_restating_the_builtin_agrees(bk, kernel, injected):
    rng = np.random.default_rng(3)
    D, M, T, k = 6, 300, 4, 3
    m0, p0, mu, pl = np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D)
    th0 = rng.normal(size=(M, D))
    zs, au, ru = _streams(rng, T, M, k, D)
    kern = KERNELS[kernel]
    runs = []
    for dm in (uc.gpl(bk, m0, p0, mu, pl), bk.GaussPriorLik(m0, p0, mu, pl, dtype=torch.float64)):
        smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, _dev_kernel(bk, kern), resample="systematic", seed=11, moves=k)
        if isinstance(dm, bk.CudaPriorLikModel):
            assert "bk_user_smc_" in smc.compile_log and "_moves" in smc.compile_log
        if injected:
            _inject(smc, T, zs, au, ru, True)
        else:
            smc.run()
        runs.append((np_(smc.last_indices), np_(smc.thetas), np_(smc.last_accept)))
    (iu, tu, au_), (ib, tb, ab) = runs
    assert np.array_equal(iu, ib) and np.array_equal(au_, ab)
    np.testing.assert_allclose(tu, tb, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_walk_proposal_equals_metropolis_kernel(bk, dtype):
    rng = np.random.default_rng(4)
    D, M, T, k, s = 5, 2000, 5, 3, 0.3
    m0, p0, mu, pl = np.zeros(D), np.ones(D), rng.normal(size=D), 4 * np.ones(D)
    th0 = rng.normal(size=(M, D))
    model = uc.gpl(bk, m0, p0, mu, pl, dtype=dtype)
    prop = bk.CudaProposal(uc.WALK, D, params=[s], transition=False, dtype=dtype)
    a = bk.TemperedLikelihoodSMC(model, M, T, th0, bk.proposal_kernel(prop), resample="systematic", seed=5, moves=k)
    assert "bk_user_smc_mhp_moves" in a.compile_log
    b = bk.TemperedLikelihoodSMC(model, M, T, th0, bk.metropolis_kernel(s), resample="systematic", seed=5, moves=k)
    a.run()
    b.run()
    assert torch.equal(a.last_indices, b.last_indices) and torch.equal(a.thetas, b.thetas)
    assert torch.equal(a.last_accept, b.last_accept) and int(a.last_accept.max()) > 1


@pytest.mark.parametrize("world", [2, 3, 5])
def test_sharded_equals_single_rank_and_oracle(bk, world):
    rng = np.random.default_rng(9)
    D, M, T, k = 6, 257, 4, 3
    dm, nm, _ = _models(bk, "gpl6", rng)
    th0 = rng.normal(size=(M, D))
    zs, au, ru = _streams(rng, T, M, k, D)
    oth, oidx, _ = mo.smc_tempered(nm, th0, zs, au, ru, T, ("rw", 0.4), resample="systematic")

    def make(group):
        return bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.metropolis_kernel(0.4), resample="systematic", group=group,
                                        moves=k, seed=13)
    inj = lambda n, lo, hi, s: (zs[n - 1, lo:hi], au[n - 1, lo:hi], ru[n - 1, :1])
    idx1, th1, _ = uc.run_fake(bk, 1, make, T, inj)
    idxg, thg, _ = uc.run_fake(bk, world, make, T, inj)
    assert np.array_equal(idx1, oidx) and np.array_equal(idxg, oidx)
    np.testing.assert_allclose(th1, oth, rtol=1e-12, atol=1e-12)
    assert np.array_equal(thg, th1)
    # Philox: the result does not depend on the world size
    none = lambda n, lo, hi, s: (None, None, None)
    p1, q1, _ = uc.run_fake(bk, 1, make, T, none)
    pg, qg, _ = uc.run_fake(bk, world, make, T, none)
    assert np.array_equal(p1, pg) and np.array_equal(q1, qg)


@pytest.mark.parametrize("thr", [0.5, 0.9])
def test_adaptive_resampling_with_moves_matches_the_oracle(bk, thr):
    rng = np.random.default_rng(11)
    D, M, T, k, s = 5, 300, 10, 2, 0.3
    dm, nm, _ = _models(bk, "gpl5", rng)
    th0 = rng.normal(size=(M, D))
    zs, au, ru = _streams(rng, T, M, k, D)
    oth, ologw, oflags = mo.smc_tempered_adaptive(nm, th0, zs, au, ru, T, thr, ("rw", s))
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, bk.metropolis_kernel(s), resample="systematic", ess_threshold=thr,
                                   moves=k)
    _inject(smc, T, zs, au, ru, True)
    assert smc.resampled == list(oflags)
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(np_(smc.log_weights), ologw, rtol=1e-10, atol=1e-12)


def test_run_steps_and_transition_mix(bk):
    D, M, T, k = 50, 4096, 6, 4
    g = torch.Generator(device="cuda").manual_seed(2)
    mu = torch.randn(D, device="cuda", generator=g)
    th0 = torch.randn(M, D, device="cuda", generator=g)
    model = bk.GaussPriorLik(torch.zeros(D), torch.ones(D), mu, 4 * torch.ones(D))
    make = lambda: bk.TemperedLikelihoodSMC(model, M, T, th0, bk.metropolis_kernel(0.2), resample="systematic",
                                            seed=21, moves=k)
    a, b = make(), make()
    for n in range(1, T + 1):
        a.transition(n)
    b.run_steps(1, 2)
    b.transition(3)
    b.run_steps(4, T)
    assert torch.equal(a.thetas, b.thetas) and torch.equal(a.last_indices, b.last_indices)
    assert torch.equal(a.last_accept, b.last_accept)


def test_more_moves_reach_the_posterior(bk):
    """fp32, Philox, seed 3: GaussPriorLik D = 50, m0 = 0, p0 = 1, pl = 4 (posterior N(0.8 mu, 0.2 I)), M = 2^16,
    T = 20, RW 0.2, systematic resampling.  A vectorised NumPy run of the same algorithm (NumPy streams, seeds 0, 1, 2,
    mu from default_rng(0)) gave a max-abs posterior-mean error of 0.43 / 0.81 / 0.89 with moves = 1 and
    0.0105 / 0.0085 / 0.0060 with moves = 20; the bound is about three times the largest moves = 20 error."""
    D, M, T = 50, 1 << 16, 20
    mu = np.random.default_rng(0).normal(size=D)
    th0 = np.random.default_rng(1).normal(size=(M, D))
    model = bk.GaussPriorLik(np.zeros(D), np.ones(D), mu, 4 * np.ones(D), dtype=torch.float32)
    err = {}
    for k in (1, 20):
        smc = bk.TemperedLikelihoodSMC(model, M, T, th0, bk.metropolis_kernel(0.2), resample="systematic", seed=3,
                                       moves=k)
        smc.run()
        err[k] = float(np.abs(np_(smc.thetas).astype(np.float64).mean(0) - 0.8 * mu).max())
    assert err[20] < 0.03
    assert err[1] > 5 * err[20]


@pytest.mark.parametrize("kernel", ["rw", "mala"])
def test_philox_moves_read_move_zero_words_at_the_block_offset(bk, kernel):
    """fp64, device Philox: move j of temperature n reads move 0's words at element block b + 2^16 j -- the normals
    and the accept uniform -- rebuilt here by the NumPy Philox and fed to the composed-kernel restatement."""
    from oracle import philox as ph
    rng = np.random.default_rng(12)
    D, M, T, k, seed = 6, 64, 3, 3, 0x5EED1234
    dm, nm, _ = _models(bk, "gpl6", rng)
    th0 = rng.normal(size=(M, D))
    ch = np.arange(M, dtype=np.uint64)
    nb = ph.accept_block(D)
    zs, au, ru = np.empty((T, M, k, D)), np.empty((T, M, k)), np.empty((T, M))
    for n in range(1, T + 1):
        for j in range(k):
            off = mo.smc_move_block(j)
            z4 = np.stack([ph.normal4_f64(seed, b + off, ch, n) for b in range(nb)])   # [nb, 4, M]
            zs[n - 1, :, j] = np.moveaxis(z4, 2, 0).reshape(M, 4 * nb)[:, :D]
            w = ph.gen(seed, nb + off, ph.TAG_NORMAL, ch, n)
            au[n - 1, :, j] = ph.u01d(w[0], w[1])
        ru[n - 1] = ph.philox_uniform(seed, 0, 0, n, np.float64, tag=ph.TAG_RESAMPLE)
    kern = KERNELS[kernel]
    oth, oidx, oacc = mo.smc_tempered(nm, th0, zs, au, ru, T, kern, resample="systematic")
    smc = bk.TemperedLikelihoodSMC(dm, M, T, th0, _dev_kernel(bk, kern), resample="systematic", seed=seed, moves=k)
    smc.run()
    assert np.array_equal(np_(smc.last_indices), oidx[-1])
    assert np.array_equal(np_(smc.last_accept), oacc[-1])
    np.testing.assert_allclose(np_(smc.thetas), oth, rtol=1e-10, atol=1e-10)
