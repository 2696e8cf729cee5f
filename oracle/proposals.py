"""NumPy restatement of Metropolis(-Hastings) with a user-written proposal (``CudaProposal``) and of the proposal's
device random streams (``proposal_normal_block`` in ``bayes-kit_b200/csrc/device_rng.cuh``).

TEST INFRASTRUCTURE (see oracle/__init__.py).

``metropolis_hastings`` follows ``MetropolisHastings.sample / _propose / _accept_test`` (metropolis.py:107-135) with a
caller-supplied proposal, driven by injected streams like the samplers of ``oracle.samplers``; ``*_batch`` loops it
over a leading chain axis.  The stream helpers rebuild the Philox-mode streams of a proposal from ``oracle.philox``.
"""
from __future__ import annotations

import numpy as np

from .philox import accept_block, philox_uniform
from .samplers import _log_u, _stack_chains


def metropolis_hastings(model, theta0, normals, uniforms, propose, transition=None, with_ratio=False):
    """Metropolis(-Hastings) with a caller-supplied proposal for one chain.

    ``propose(theta, z, u) -> theta'`` and ``transition(to, frm) -> log q(to | frm)`` are NumPy restatements of a
    ``CudaProposal``.  normals: [n, n_normals]; uniforms: [n, 1 + n_uniforms] (or [n] without proposal uniforms),
    column 0 the accept uniform and columns 1.. the proposal's ``u``.  ``transition=None`` is ``Metropolis``
    (metropolis.py:12-38); otherwise the Hastings test of metropolis.py:41-76 with
    ``fwd = transition(proposal, theta)``, ``rev = transition(theta, proposal)``.  Returns (draws [n, D], logp [n],
    accepted [n] bool) (, log ratio [n] with ``with_ratio``)."""
    theta = np.array(theta0, dtype=np.float64, copy=True)
    n, dim = normals.shape[0], theta.shape[0]
    uniforms = np.asarray(uniforms, dtype=np.float64).reshape(n, -1)
    lp = model.log_density(theta)
    ratios = np.empty(n)
    draws = np.empty((n, dim))
    logps = np.empty(n)
    acc = np.zeros(n, dtype=bool)
    for t in range(n):
        prop = np.asarray(propose(theta, normals[t], uniforms[t, 1:]), dtype=np.float64)
        lp_p = model.log_density(prop)
        ratio = lp_p - lp
        if transition is not None:
            fwd = transition(prop, theta)
            rev = transition(theta, prop)
            ratio = ratio + (rev - fwd)
        ratios[t] = ratio
        if _log_u(uniforms[t, 0]) < ratio:
            theta, lp = prop, lp_p
            acc[t] = True
        draws[t] = theta
        logps[t] = lp
    return (draws, logps, acc, ratios) if with_ratio else (draws, logps, acc)


def metropolis_hastings_batch(model, theta0, normals, uniforms, propose, transition=None, with_ratio=False):
    """theta0 [C, D], normals [n, C, n_normals], uniforms [n, C, 1 + n_uniforms] ->
    draws [n, C, D], logp [n, C], acc [n, C] (, log ratio [n, C])."""
    C = theta0.shape[0]
    return _stack_chains([metropolis_hastings(model, theta0[c], normals[:, c], uniforms[:, c], propose, transition,
                                              with_ratio) for c in range(C)])


# ---- Philox-mode streams of a proposal ----------------------------------------------------------------------------
def proposal_normal_block(k, D):
    """``proposal_normal_block``: element block of a user proposal's normal k -- k // 4, skipping accept_block(D)."""
    b = np.asarray(k, dtype=np.int64) >> 2
    return np.where(b < accept_block(D), b, b + 1)


def proposal_blocks(D, n_normals):
    """The element blocks whose normals make up a proposal's z[0 .. n_normals), in order."""
    return [int(proposal_normal_block(4 * j, D)) for j in range((int(n_normals) + 3) // 4)]


def proposal_uniforms(seed, chain_offset, draw, C, n_uniforms, dtype=np.float64):
    """[C, n_uniforms]: u[k] of a user proposal, the k-th TAG_UNIFORM uniform of (global chain, draw)."""
    k = np.arange(int(n_uniforms), dtype=np.uint64)[None, :]
    ch = (np.uint64(chain_offset) + np.arange(C, dtype=np.uint64))[:, None]
    return philox_uniform(seed, k, ch, draw, dtype).reshape(C, int(n_uniforms))
