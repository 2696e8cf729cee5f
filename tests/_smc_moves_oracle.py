"""NumPy restatement of TemperedLikelihoodSMC with several Markov moves per temperature (``moves=k``).

It builds on ``oracle.samplers`` and ``_smc_proposal_oracle``. The weights, both resamplers and the single move are
those modules'. Only the move changes: each particle gets k applications of the kernel at time(n-1), in stream order,
before it is reweighted to time(n) and resampled. This is the reference run with the composed kernel
``K(K(...K(theta)))``. Streams are ``[T, M, k, ...]``: normals ``[T, M, k, D]`` (proposal move:
``[T, M, k, n_normals]``) and accept uniforms ``[T, M, k]`` (proposal move: ``[T, M, k]`` or
``[T, M, k, 1 + n_uniforms]``). The random-walk, MALA and HMC moves of ``oracle.samplers.smc_move`` do not report
their decision. A move counts as accepted when it changes the particle, which is the decision whenever the proposal
differs from the current point (any non-zero normal)."""
import numpy as np

import _smc_proposal_oracle as sop
from oracle import samplers as osm


def smc_move_block(j):
    """Offset of the element-block counter word for move j of a temperature step (device_rng.cuh smc_move_block):
    move j draws exactly move 0's Philox words at block b + 2^16 j."""
    return int(j) << 16


def _resample(model, thetas, n, T, ru, resample):
    """indices of importance_resample at step n, as oracle.samplers.smc_tempered forms them"""
    if resample == "multinomial":
        idx, _ = osm.multinomial_indices(osm.smc_weights(model, thetas, n, T), ru)
        return idx
    t0, t1 = (n - 1) / T, n / T
    logw = np.array([(model.log_likelihood(th) * t1 + model.log_prior(th)) -
                     (model.log_likelihood(th) * t0 + model.log_prior(th)) for th in thetas])
    idx, _ = osm.systematic_indices(logw, ru[0])
    return idx


def _composed(move, thetas, zs, us):
    """every particle through its k moves -> accepted moves per particle"""
    acc = np.zeros(thetas.shape[0], dtype=np.int64)
    for m in range(thetas.shape[0]):
        for j in range(zs.shape[1]):
            new, a = move(thetas[m], zs[m, j], us[m, j])
            thetas[m] = new
            acc[m] += a
    return acc


def _kernel_move(model, t0, kernel):
    def move(th, z, u):
        new = osm.smc_move(model, th, t0, z, u, kernel)
        return new, int(not np.array_equal(new, th))
    return move


def smc_tempered(model, thetas0, prop_normals, acc_uniforms, res_uniforms, T, kernel, resample="multinomial"):
    """``oracle.samplers.smc_tempered`` with k = prop_normals.shape[2] moves per temperature.  kernel: as
    ``oracle.samplers.smc_move`` takes it.  Returns (thetas_final [M, D], idx [T, M], accepted moves [T, M])."""
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    all_idx = np.empty((T, M), dtype=np.int64)
    all_acc = np.empty((T, M), dtype=np.int64)
    for n in range(1, T + 1):
        all_acc[n - 1] = _composed(_kernel_move(model, (n - 1) / T, kernel), thetas, prop_normals[n - 1],
                                   acc_uniforms[n - 1])
        idx = _resample(model, thetas, n, T, res_uniforms[n - 1], resample)
        all_idx[n - 1] = idx
        thetas = thetas[idx]
    return thetas, all_idx, all_acc


def smc_tempered_adaptive(model, thetas0, prop_normals, acc_uniforms, res_uniforms, T, ess_threshold, kernel):
    """``oracle.samplers.smc_tempered_adaptive`` with k moves per temperature.  Returns (thetas, logw, resampled [T])."""
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    logw = np.zeros(M)
    flags = np.zeros(T, dtype=bool)
    lp = lambda th, t: model.log_likelihood(th) * t + model.log_prior(th)
    for n in range(1, T + 1):
        t0, t1 = (n - 1) / T, n / T
        _composed(_kernel_move(model, t0, kernel), thetas, prop_normals[n - 1], acc_uniforms[n - 1])
        logw = logw + np.array([lp(th, t1) - lp(th, t0) for th in thetas])
        wi, _ = osm.systematic_weights(logw)
        wf = wi.astype(np.float64)
        if float(int(wi.sum())) ** 2 / (wf ** 2).sum() < ess_threshold * M:
            idx, _ = osm.systematic_indices(logw, res_uniforms[n - 1, 0])
            thetas, logw, flags[n - 1] = thetas[idx], np.zeros(M), True
    return thetas, logw, flags


def smc_tempered_proposal(model, thetas0, normals, acc_uniforms, res_uniforms, T, propose, transition=None,
                          resample="multinomial"):
    """``_smc_proposal_oracle.smc_tempered`` with k moves per temperature.  The accept decisions are the proposal
    move's own.  Returns (thetas_final [M, D], idx [T, M], accepted moves [T, M])."""
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    all_idx = np.empty((T, M), dtype=np.int64)
    all_acc = np.empty((T, M), dtype=np.int64)
    for n in range(1, T + 1):
        t0 = (n - 1) / T
        move = lambda th, z, u: sop.smc_move(model, th, t0, z, u, propose, transition)
        all_acc[n - 1] = _composed(move, thetas, normals[n - 1], acc_uniforms[n - 1])
        idx = _resample(model, thetas, n, T, res_uniforms[n - 1], resample)
        all_idx[n - 1] = idx
        thetas = thetas[idx]
    return thetas, all_idx, all_acc
