"""NumPy restatement of the reference samplers, driven by *injected* RNG streams.

TEST INFRASTRUCTURE (see oracle/__init__.py).

Each function advances ONE chain (the reference has no multi-chain driver:
one sampler object == one chain, SURVEY.md section 1) and consumes pre-drawn
standard normals / uniforms in the reference's consumption order instead of
owning a generator.  ``*_batch`` helpers loop the single-chain function over a
leading chain axis; that is what the CUDA kernels are diffed against.

The elementwise arithmetic is written in the reference's association order so
fp64 results agree to rounding with the unmodified reference
(``oracle/gen_golden.py`` checks this against the live reference).
"""
from __future__ import annotations

import math

import numpy as np


def _as_metric(metric, dim):
    # reference: ``metric_diag or np.ones(dim)`` (hmc.py:22, drghmc.py:70)
    return np.ones(dim) if metric is None else np.asarray(metric, dtype=np.float64)


# --------------------------------------------------------------------------
# HMCDiag  -- bayes_kit/hmc.py
# --------------------------------------------------------------------------
def hmc_diag(model, theta0, normals, uniforms, stepsize, steps, metric=None, with_ratio=False):
    """n draws of diagonal-metric HMC for one chain.

    Follows ``HMCDiag.sample`` (hmc.py:55-63), ``joint_logp`` (hmc.py:36-38)
    and ``leapfrog`` (hmc.py:40-53): backward half kick, ``steps`` x
    {full kick, drift, gradient}, forward half kick; accept iff
    ``log(u) < H1 - H0`` (strict); returns the *joint* log density.

    normals: [n, D] momentum draws; uniforms: [n] accept uniforms.
    Returns (draws [n, D], logp [n], accepted [n] bool), and with ``with_ratio``
    the log acceptance ratio H1 - H0 [n] the accept test compared ``log(u)`` with.
    """
    theta = np.array(theta0, dtype=np.float64, copy=True)
    n, dim = normals.shape
    m = _as_metric(metric, dim)
    ratio = np.empty(n)
    half = 0.5 * stepsize
    draws = np.empty((n, dim))
    logps = np.empty(n)
    acc = np.zeros(n, dtype=bool)
    for t in range(n):
        rho = normals[t]
        h0 = model.log_density(theta) - 0.5 * np.dot(rho, m * rho)
        _, g = model.log_density_gradient(theta)
        g = np.asarray(g)
        q = theta
        r = rho - half * (m * g)
        for _ in range(steps):
            r = r + stepsize * (m * g)
            q = q + stepsize * r
            _, g = model.log_density_gradient(q)
            g = np.asarray(g)
        r = r + half * (m * g)
        h1 = model.log_density(q) - 0.5 * np.dot(r, m * r)
        ratio[t] = h1 - h0
        if _log_u(uniforms[t]) < h1 - h0:
            theta = q
            logps[t] = h1
            acc[t] = True
        else:
            logps[t] = h0
        draws[t] = theta
    return (draws, logps, acc, ratio) if with_ratio else (draws, logps, acc)


# --------------------------------------------------------------------------
# MALA  -- bayes_kit/mala.py
# --------------------------------------------------------------------------
def mala(model, theta0, normals, uniforms, epsilon, with_ratio=False):
    """n MALA draws for one chain.

    Follows ``MALA.sample`` (mala.py:40-66) with the cached (lp, grad) of the
    current point (mala.py:31-32, 62-64), the proposal density
    ``q(a|b) = -(1/4eps) |a - b - eps grad_b|^2`` (mala.py:68-79) and the
    Metropolis-Hastings test of metropolis.py:41-76.  ``with_ratio``: also
    return the log acceptance ratio [n] (as hmc_diag).
    """
    theta = np.array(theta0, dtype=np.float64, copy=True)
    n, dim = normals.shape
    lp, g = model.log_density_gradient(theta)
    g = np.asarray(g)
    sd = np.sqrt(2 * epsilon)
    coef = -0.25 / epsilon
    ratio = np.empty(n)
    draws = np.empty((n, dim))
    logps = np.empty(n)
    acc = np.zeros(n, dtype=bool)
    for t in range(n):
        prop = theta + epsilon * g + sd * normals[t]
        lp_p, g_p = model.log_density_gradient(prop)
        g_p = np.asarray(g_p)
        d_f = prop - theta - epsilon * g
        d_r = theta - prop - epsilon * g_p
        fwd = coef * d_f.dot(d_f)
        rev = coef * d_r.dot(d_r)
        log_ratio = (lp_p - lp) + (rev - fwd)
        ratio[t] = log_ratio
        if _log_u(uniforms[t]) < log_ratio:
            theta, lp, g = prop, lp_p, g_p
            acc[t] = True
        draws[t] = theta
        logps[t] = lp
    return (draws, logps, acc, ratio) if with_ratio else (draws, logps, acc)


def _log_u(u):
    # np.log(0.0) == -inf in the reference (a RuntimeWarning, not an error)
    return math.log(u) if u > 0 else -math.inf


# --------------------------------------------------------------------------
# Metropolis / MetropolisHastings with a Gaussian random-walk proposal
# -- bayes_kit/metropolis.py
# --------------------------------------------------------------------------
def metropolis_rw(model, theta0, normals, uniforms, scale, hastings=False, with_ratio=False):
    """Random-walk Metropolis: proposal ``theta + scale * z``.

    Follows ``MetropolisHastings.sample/_propose/_accept_test``
    (metropolis.py:107-135) with ``proposal_fn = normal(loc=theta, scale)`` and
    the accept rules of metropolis.py:12-38 / 41-76.  With ``hastings=True`` the
    (exactly cancelling) symmetric transition terms are included, as
    ``MetropolisHastings`` would compute them.  ``with_ratio``: also return the
    log acceptance ratio [n] (as hmc_diag).
    """
    theta = np.array(theta0, dtype=np.float64, copy=True)
    n, dim = normals.shape
    lp = model.log_density(theta)
    ratios = np.empty(n)
    draws = np.empty((n, dim))
    logps = np.empty(n)
    acc = np.zeros(n, dtype=bool)
    for t in range(n):
        prop = theta + scale * normals[t]
        lp_p = model.log_density(prop)
        ratio = lp_p - lp
        if hastings:
            d = prop - theta
            fwd = -0.5 * np.dot(d, d) / (scale * scale)
            d2 = theta - prop
            rev = -0.5 * np.dot(d2, d2) / (scale * scale)
            ratio = ratio + (rev - fwd)
        ratios[t] = ratio
        if _log_u(uniforms[t]) < ratio:
            theta, lp = prop, lp_p
            acc[t] = True
        draws[t] = theta
        logps[t] = lp
    return (draws, logps, acc, ratios) if with_ratio else (draws, logps, acc)


# --------------------------------------------------------------------------
# DrGhmcDiag  -- bayes_kit/drghmc.py
# --------------------------------------------------------------------------
class _DrState:
    """Explicit (logp, grad) stack standing in for the reference's
    ``_log_density_gradient_cache`` (drghmc.py:82, 243-247, 276, 288)."""

    def __init__(self, model, metric, sizes, counts, prob_retry):
        self.model = model
        self.m = metric
        self.sizes = sizes
        self.counts = counts
        self.prob_retry = bool(prob_retry)
        self.stack = []
        self.n_grad = 0

    def grad(self, q):
        self.n_grad += 1
        lp, g = self.model.log_density_gradient(q)
        return lp, np.asarray(g, dtype=np.float64)

    def kinetic(self, r):
        return 0.5 * np.dot(r, self.m * r)

    def retry(self, reject_logp):
        # drghmc.py:317 -- bool * float (False * -inf is nan, on purpose)
        return self.prob_retry * reject_logp

    def propose(self, q, r, k):
        """leapfrog (drghmc.py:253-289) + momentum flip (drghmc.py:319-346).
        Starts from the gradient on top of the stack, pushes the endpoint."""
        eps, cnt = self.sizes[k], self.counts[k]
        q = np.array(q, copy=True)
        _, g = self.stack[-1]
        r = r + 0.5 * eps * (self.m * g)
        q += eps * r
        for _ in range(cnt - 1):
            _, g = self.grad(q)
            r += eps * (self.m * g)
            q += eps * r
        lp, g = self.grad(q)
        r = r + 0.5 * eps * (self.m * g)
        self.stack.append((lp, g))
        return q, -r

    def log_accept(self, q_p, r_p, k, cur_hastings, cur_logp):
        """drghmc.py:391-446: joint density of the proposal (from the stack
        top), ghost proposals i<k started at the proposal, Hastings + retry
        terms, ``min(0, .)`` with Python semantics (nan -> 0)."""
        prop_logp = self.stack[-1][0] - self.kinetic(r_p)
        prop_hastings = 0
        for i in range(k):
            q_g, r_g = self.propose(q_p, r_p, i)
            a, _ = self.log_accept(q_g, r_g, i, prop_hastings, prop_logp)
            self.stack.pop()
            if a == 0:
                return -np.inf, prop_logp
            prop_hastings += np.log1p(-np.exp(a))
        frac = (
            (prop_logp - cur_logp)
            + (prop_hastings - cur_hastings)
            + (self.retry(prop_hastings) - self.retry(cur_hastings))
        )
        return (frac if frac < 0 else 0), prop_logp


def drghmc(model, theta0, rho0, normals, uniforms, max_proposals, step_sizes,
           step_counts, damping, metric=None, prob_retry=True):
    """n DrGhmcDiag draws for one chain (drghmc.py:348-389).

    normals: [n, D] refresh normals; uniforms: [n, 2K] in consumption order
    (retry test then accept test per attempt, drghmc.py:370,378); unused slots
    may hold anything.  Returns (draws, joint logp, rho_final, n_uniforms_used
    [n], n_grad_evals).
    """
    theta = np.array(theta0, dtype=np.float64, copy=True)
    rho = np.array(rho0, dtype=np.float64, copy=True)
    n, dim = normals.shape
    st = _DrState(model, _as_metric(metric, dim), list(step_sizes),
                  list(step_counts), prob_retry)
    draws = np.empty((n, dim))
    logps = np.empty(n)
    used = np.zeros(n, dtype=np.int64)
    with np.errstate(all="ignore"):
        for t in range(n):
            rho = rho * np.sqrt(1 - damping) + np.sqrt(damping) * normals[t]
            if not st.stack:
                st.stack = [st.grad(theta)]
            cur_logp = st.stack[-1][0] - st.kinetic(rho)
            cur_hastings, reject_logp = 0.0, 0.0
            ui = 0
            for k in range(max_proposals):
                u = uniforms[t, ui]; ui += 1
                if not (_log_u(u) < st.retry(reject_logp)):
                    break
                q_p, r_p = st.propose(theta, rho, k)
                a, prop_logp = st.log_accept(q_p, r_p, k, cur_hastings, cur_logp)
                u = uniforms[t, ui]; ui += 1
                if _log_u(u) < a:
                    theta, rho, cur_logp = q_p, r_p, prop_logp
                    break
                reject_logp = np.log1p(-np.exp(a))
                cur_hastings += reject_logp
                st.stack.pop()
            st.stack = [st.stack[-1]]
            rho = -rho
            draws[t] = theta
            logps[t] = cur_logp
            used[t] = ui
    return draws, logps, rho, used, st.n_grad


# --------------------------------------------------------------------------
# TemperedLikelihoodSMC  -- bayes_kit/smc.py
# --------------------------------------------------------------------------
def smc_weights(model, thetas, n, T):
    """``exp(lp - lpminus1)`` exactly as importance_resample evaluates it
    (smc.py:47-51, 67-70): both tempered densities in full, no max-shift."""
    t0, t1 = (n - 1) / T, n / T
    w = np.empty(thetas.shape[0])
    for i, th in enumerate(thetas):
        ll, pr = model.log_likelihood(th), model.log_prior(th)
        w[i] = (ll * t1 + pr) - (ll * t0 + pr)
    return np.exp(w)


def multinomial_indices(weights, uniforms):
    """Legacy ``np.random.choice(M, M, True, p)`` (smc.py:73) ==
    searchsorted(cumsum(p)/cumsum(p)[-1], U, 'right')  (SURVEY.md 2.1-9)."""
    p = weights / weights.sum()
    cdf = p.cumsum()
    cdf /= cdf[-1]
    return cdf.searchsorted(uniforms, side="right").astype(np.int64), cdf


def systematic_weights(logw):
    """Fixed-point importance weights of the systematic mode: w_i = rint(exp(logw_i - max) * 2^s) as int64,
    s = 61 - ceil(log2 M) (so that sum w < 2^62).  Integer sums are exact and associative: the CDF, and
    with it every resample index, is independent of how the particles are sharded over GPUs."""
    logw = np.asarray(logw, dtype=np.float64)
    M = logw.shape[0]
    lg = 0
    while (1 << lg) < M:
        lg += 1
    s = 61 - lg
    e = np.exp(logw - np.max(logw))
    e = np.where(np.isnan(e), 0.0, e)
    return np.rint(np.ldexp(e, s)).astype(np.int64), s


def systematic_indices(logw, u0):
    """Systematic resampling with a log-sum-exp normaliser (north_star item 2;
    NOT in the reference -- parity unpinned, this restatement is the oracle).
    Point k has threshold t_k = floor((k + u0) * (W / M)) in fixed-point CDF units (W = sum w, fp64
    operations in exactly this order, the rate W / M formed once, clamped to W - 1) and selects the first particle whose
    inclusive integer cumsum exceeds t_k."""
    w, _ = systematic_weights(logw)
    M = w.shape[0]
    cum = np.cumsum(w)
    W = int(cum[-1])
    t = np.floor((np.arange(M) + u0) * (float(W) / M)).astype(np.int64)
    t = np.minimum(t, W - 1)
    idx = np.searchsorted(cum, t, side="right")
    return np.minimum(idx, M - 1).astype(np.int64), cum


def smc_move(model, theta, t0, z, u, kernel):
    """One application of the SMC's Markov kernel at temperature t0 to one particle.
    kernel = ("rw", scale): metropolis_kernel (smc.py:79-89);
             ("mala", eps): one MALA.sample() on the tempered density (mala.py:40-66);
             ("hmc", eps, L): one HMCDiag.sample(), identity metric (hmc.py:40-63) -- the MCMC-kernel
             plug-ins of the TODO at smc.py:78, pinned by gen_golden.py against the reference's own MALA /
             HMCDiag classes driven on the tempered model."""
    from .models import Tempered
    kind = kernel[0]
    if kind == "rw":
        lp = lambda th: model.log_likelihood(th) * t0 + model.log_prior(th)
        star = theta + kernel[1] * z
        return star if _log_u(u) < lp(star) - lp(theta) else theta
    tm = Tempered(model, t0)
    if kind == "mala":
        d, _, _ = mala(tm, theta, z[None], np.array([u]), kernel[1])
        return d[0]
    if kind == "hmc":
        d, _, _ = hmc_diag(tm, theta, z[None], np.array([u]), kernel[1], kernel[2])
        return d[0]
    raise ValueError(kind)


def smc_tempered(model, thetas0, prop_normals, acc_uniforms, res_uniforms,
                 scale, T, resample="multinomial", kernel=None):
    """Full run of TemperedLikelihoodSMC.

    ``run``/``transition`` (smc.py:39-60): for n = 1..T move every particle
    once with the kernel (default ``metropolis_kernel(scale)``, smc.py:79-89) targeting the
    PREVIOUS temperature, then reweight to ``time(n)`` and resample.
    prop_normals [T, M, D], acc_uniforms [T, M], res_uniforms [T, M]
    (systematic: only res_uniforms[:, 0] is used).
    Returns (thetas_final [M, D], idx [T, M]).
    """
    kernel = ("rw", scale) if kernel is None else kernel
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    all_idx = np.empty((T, M), dtype=np.int64)
    for n in range(1, T + 1):
        t0 = (n - 1) / T

        def lpm1(th):
            return model.log_likelihood(th) * t0 + model.log_prior(th)

        for m in range(M):
            thetas[m] = smc_move(model, thetas[m], t0, prop_normals[n - 1, m], acc_uniforms[n - 1, m], kernel)
        if resample == "multinomial":
            w = smc_weights(model, thetas, n, T)
            idx, _ = multinomial_indices(w, res_uniforms[n - 1])
        else:
            t1 = n / T
            logw = np.array([
                (model.log_likelihood(th) * t1 + model.log_prior(th)) - lpm1(th)
                for th in thetas])
            idx, _ = systematic_indices(logw, res_uniforms[n - 1, 0])
        all_idx[n - 1] = idx
        thetas = thetas[idx]
    return thetas, all_idx


# --------------------------------------------------------------------------
# batch helpers (leading chain axis)
# --------------------------------------------------------------------------
def _stack_chains(out):
    return tuple(np.stack([o[i] for o in out], 1) for i in range(len(out[0])))


def hmc_diag_batch(model, theta0, normals, uniforms, stepsize, steps, metric=None, with_ratio=False):
    """theta0 [C, D], normals [n, C, D], uniforms [n, C] ->
    draws [n, C, D], logp [n, C], acc [n, C] (, log ratio [n, C])."""
    C = theta0.shape[0]
    return _stack_chains([hmc_diag(model, theta0[c], normals[:, c], uniforms[:, c], stepsize,
                                   steps, metric, with_ratio) for c in range(C)])


def mala_batch(model, theta0, normals, uniforms, epsilon, with_ratio=False):
    C = theta0.shape[0]
    return _stack_chains([mala(model, theta0[c], normals[:, c], uniforms[:, c], epsilon, with_ratio)
                          for c in range(C)])


def metropolis_rw_batch(model, theta0, normals, uniforms, scale, hastings=False, with_ratio=False):
    C = theta0.shape[0]
    return _stack_chains([metropolis_rw(model, theta0[c], normals[:, c], uniforms[:, c], scale,
                                        hastings, with_ratio) for c in range(C)])


def drghmc_batch(model, theta0, rho0, normals, uniforms, max_proposals,
                 step_sizes, step_counts, damping, metric=None, prob_retry=True):
    """theta0/rho0 [C, D], normals [n, C, D], uniforms [n, C, 2K]."""
    C = theta0.shape[0]
    out = [drghmc(model, theta0[c], rho0[c], normals[:, c], uniforms[:, c],
                  max_proposals, step_sizes, step_counts, damping, metric,
                  prob_retry) for c in range(C)]
    return (np.stack([o[0] for o in out], 1), np.stack([o[1] for o in out], 1),
            np.stack([o[2] for o in out], 0), np.stack([o[3] for o in out], 1))


# ---- Stretcher (ensemble.py:9-66) -- PARITY UNPINNED --------------------------------
# Upstream the whole implementation is commented out, so there is no executable
# reference: this is a restatement of the algorithm its comments sketch (Goodman &
# Weare 2010), with the three uniforms of a move injected so the device kernel can be
# compared draw for draw.  Conventions fixed here (the sketch leaves them open):
# partner j = floor(u0 * m); z = (1/sqrt(a) + (sqrt(a) - 1/sqrt(a)) * u1) ** 2
# (ensemble.py:43-46); accept iff log(u2) < (D-1) log z + lp(theta*) - lp(theta_k) (:48-53).
def stretch_half(model, active, other, u, a=2.0):
    """Move every walker of `active` [n, D] against `other` [m, D]; u [n, 3].
    Returns (new_active, accepted [n] bool, logp of the new walkers)."""
    active = np.array(active, dtype=np.float64, copy=True)
    other = np.asarray(other, dtype=np.float64)
    n, D = active.shape
    m = other.shape[0]
    lo, hi = 1.0 / np.sqrt(a), np.sqrt(a)
    acc = np.zeros(n, dtype=bool)
    lps = np.zeros(n)
    for k in range(n):
        j = min(int(u[k, 0] * m), m - 1)
        z = np.square(lo + (hi - lo) * u[k, 1])
        star = other[j] + z * (active[k] - other[j])
        lp_k, lp_s = model.log_density(active[k]), model.log_density(star)
        log_q = (D - 1) * np.log(z) + lp_s - lp_k
        if _log_u(u[k, 2]) < log_q:
            active[k], acc[k], lps[k] = star, True, lp_s
        else:
            lps[k] = lp_k
    return active, acc, lps


def stretch(model, thetas0, us, a=2.0):
    """n_steps of Stretcher.sample() (ensemble.py:55-63): first half against the second,
    then the second half against the UPDATED first.  us [n_steps, W, 3] (row k of a step
    belongs to walker k).  Returns (thetas [n_steps, W, D], accepts [n_steps, W])."""
    th = np.array(thetas0, dtype=np.float64, copy=True)
    W = th.shape[0]
    h = W // 2
    out, accs = [], []
    for u in us:
        a1, acc1, _ = stretch_half(model, th[:h], th[h:], u[:h], a)
        th[:h] = a1
        a2, acc2, _ = stretch_half(model, th[h:], th[:h], u[h:], a)
        th[h:] = a2
        out.append(th.copy())
        accs.append(np.concatenate([acc1, acc2]))
    return np.stack(out), np.stack(accs)


def smc_tempered_adaptive(model, thetas0, prop_normals, acc_uniforms, res_uniforms, scale, T, ess_threshold):
    """TemperedLikelihoodSMC with ESS-triggered systematic resampling -- PARITY UNPINNED (the
    reference resamples unconditionally, smc.py:60; this is the textbook adaptive variant, SURVEY 8f-4).
    Moves as in smc_tempered; log-weights accumulate until (sum w)^2 / sum w^2 < ess_threshold * M,
    then systematic resampling with u0 = res_uniforms[n-1, 0] and the weights reset.
    Returns (thetas, logw, resampled [T] bool)."""
    thetas = np.array(thetas0, dtype=np.float64, copy=True)
    M = thetas.shape[0]
    logw = np.zeros(M)
    flags = np.zeros(T, dtype=bool)
    for n in range(1, T + 1):
        t0, t1 = (n - 1) / T, n / T
        lp = lambda th, t: model.log_likelihood(th) * t + model.log_prior(th)
        for m in range(M):
            star = thetas[m] + scale * prop_normals[n - 1, m]
            if _log_u(acc_uniforms[n - 1, m]) < lp(star, t0) - lp(thetas[m], t0):
                thetas[m] = star
        logw = logw + np.array([lp(th, t1) - lp(th, t0) for th in thetas])
        wi, _ = systematic_weights(logw)          # the ESS of the fixed-point weights the resampler uses
        wf = wi.astype(np.float64)
        if float(int(wi.sum())) ** 2 / (wf ** 2).sum() < ess_threshold * M:
            idx, _ = systematic_indices(logw, res_uniforms[n - 1, 0])
            thetas, logw, flags[n - 1] = thetas[idx], np.zeros(M), True
    return thetas, logw, flags
