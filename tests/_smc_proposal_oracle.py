"""NumPy restatement of TemperedLikelihoodSMC with a user-written proposal as the move (``proposal_kernel``).

It builds on ``oracle.samplers`` (the weights and both resamplers are that module's) and changes only the move: one
Metropolis(-Hastings) step of a caller-supplied proposal on the tempered density ``lp_t = ll * t0 + prior``, in the
order of ``oracle.proposals.metropolis_hastings``.  ``propose(theta, z, u) -> theta*`` and ``transition(to, frm) ->
log q(to | frm)`` (None: no Hastings term) are NumPy restatements of a ``CudaProposal``.  Accept uniforms are
``[T, M]`` (a proposal without uniforms) or ``[T, M, 1 + n_uniforms]``: column 0 is the accept uniform, columns 1..
the proposal's ``u``."""
import numpy as np

from oracle import samplers as osm


def smc_move(model, theta, t0, z, u, propose, transition=None):
    """One move of one particle -> (theta', accepted)."""
    u = np.atleast_1d(np.asarray(u, dtype=np.float64))
    lp = lambda th: model.log_likelihood(th) * t0 + model.log_prior(th)
    star = np.asarray(propose(theta, z, u[1:]), dtype=np.float64)
    ratio = lp(star) - lp(theta)
    if transition is not None:
        ratio = ratio + (transition(theta, star) - transition(star, theta))
    acc = bool(osm._log_u(u[0]) < ratio)
    return (star if acc else theta), acc


def _move_all(model, thetas, t0, normals, acc_uniforms, propose, transition):
    acc = np.zeros(thetas.shape[0], dtype=bool)
    for m in range(thetas.shape[0]):
        thetas[m], acc[m] = smc_move(model, thetas[m], t0, normals[m], acc_uniforms[m], propose, transition)
    return acc


def smc_tempered(model, thetas0, normals, acc_uniforms, res_uniforms, T, propose, transition=None,
                 resample="multinomial"):
    """``oracle.samplers.smc_tempered`` with the proposal move.  normals [T, M, n_normals].
    Returns (thetas_final [M, D], idx [T, M], accepted [T, M])."""
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    all_idx = np.empty((T, M), dtype=np.int64)
    all_acc = np.empty((T, M), dtype=bool)
    for n in range(1, T + 1):
        t0, t1 = (n - 1) / T, n / T
        all_acc[n - 1] = _move_all(model, thetas, t0, normals[n - 1], acc_uniforms[n - 1], propose, transition)
        if resample == "multinomial":
            idx, _ = osm.multinomial_indices(osm.smc_weights(model, thetas, n, T), res_uniforms[n - 1])
        else:
            lp = lambda th, t: model.log_likelihood(th) * t + model.log_prior(th)
            logw = np.array([lp(th, t1) - lp(th, t0) for th in thetas])
            idx, _ = osm.systematic_indices(logw, res_uniforms[n - 1, 0])
        all_idx[n - 1] = idx
        thetas = thetas[idx]
    return thetas, all_idx, all_acc


def smc_tempered_adaptive(model, thetas0, normals, acc_uniforms, res_uniforms, T, ess_threshold, propose,
                          transition=None):
    """``oracle.samplers.smc_tempered_adaptive`` with the proposal move.  Returns (thetas, logw, resampled [T])."""
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    logw = np.zeros(M)
    flags = np.zeros(T, dtype=bool)
    lp = lambda th, t: model.log_likelihood(th) * t + model.log_prior(th)
    for n in range(1, T + 1):
        t0, t1 = (n - 1) / T, n / T
        _move_all(model, thetas, t0, normals[n - 1], acc_uniforms[n - 1], propose, transition)
        logw = logw + np.array([lp(th, t1) - lp(th, t0) for th in thetas])
        wi, _ = osm.systematic_weights(logw)
        wf = wi.astype(np.float64)
        if float(int(wi.sum())) ** 2 / (wf ** 2).sum() < ess_threshold * M:
            idx, _ = osm.systematic_indices(logw, res_uniforms[n - 1, 0])
            thetas, logw, flags[n - 1] = thetas[idx], np.zeros(M), True
    return thetas, logw, flags
