"""HMCDiag -- diagonal-metric Hamiltonian Monte Carlo (reference: bayes_kit/hmc.py)."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib as L
from ._sampler import ChainSampler
from ._util import ptr, stream_ptr, to_dev


class HMCDiag(ChainSampler):
    """Same constructor as the reference (hmc.py:9-17):
    ``HMCDiag(model, stepsize, steps, metric_diag=None, init=None, seed=None)``.

    ``sample()`` returns ``(theta, joint_logp)`` exactly like hmc.py:55-63 (the
    JOINT log density ``log p(theta) - 0.5 rho.M.rho``).  One call advances all
    chains: a single fused kernel per call for iso/diagonal Gaussian plugins
    (theta, rho in registers across the L leapfrog steps) and for a
    ``CudaModel`` / ``CudaPriorLikModel`` up to 192 dims (registers up to 32,
    the trajectory in shared memory above; the latter is compiled at
    construction, ``compile_log`` holds ptxas's report, ``""`` on every other
    engine), a GEMM-gradient pipeline for the dense / regression plugins.

    ``metric_diag``: the reference only works with None or a size-1 array
    (``metric_diag or np.ones(dim)``, hmc.py:22); a full [D] metric is accepted
    here with the reference's convention (kinetic 0.5 rho.(m rho), kick
    eps m grad, drift eps rho -- hmc.py:37,46-52).
    """

    def __init__(self, model, stepsize: float, steps: int, metric_diag=None, init=None, seed=None,
                 *, chains: Optional[int] = None, chain_offset: int = 0):
        super().__init__(model, init, seed, chains, chain_offset)
        self._stepsize = float(stepsize)
        self._steps = int(steps)
        if self._steps < 0:
            raise ValueError(f"steps must be >= 0, got {steps}")
        if metric_diag is None:
            self._metric = None
        else:
            m = to_dev(metric_diag, self.dtype, self.device).reshape(-1)
            if m.numel() == 1 and self._dim > 1:
                m = m.expand(self._dim).contiguous()
            if m.numel() != self._dim:
                raise ValueError(f"metric_diag must have {self._dim} entries")
            self._metric = m
        self._prepare_wide("HMCDiag")

    def _launch(self, n, rng, out, c0=0, cn=None, cache_valid=None):
        lib = L.lib()
        self._need_grad_cache()
        cn = self._C if cn is None else cn
        wp, wn = self._ws.get(lib.bk_hmc_diag_workspace_bytes(self._model.handle, self._C))
        L.check(lib.bk_hmc_diag_sample(
            self._model.handle, self._theta[c0:].data_ptr(), self._lp[c0:].data_ptr(),
            self._grad[c0:].data_ptr(), C.byref(self._cache_valid if cache_valid is None else cache_valid), cn, self._stepsize,
            self._steps, ptr(self._metric), n, C.byref(rng), C.byref(out), wp, wn, stream_ptr(self.device)))
