"""MALA -- Metropolis-adjusted Langevin (reference: bayes_kit/mala.py)."""
from __future__ import annotations

import ctypes as C
from typing import Optional

from . import _lib as L
from ._sampler import ChainSampler
from ._util import stream_ptr


class MALA(ChainSampler):
    """``MALA(model, epsilon, init=None, seed=None)`` (mala.py:15-21).  Proposal
    ``theta + eps grad + sqrt(2 eps) z`` (mala.py:41-45), Hastings-corrected
    accept (mala.py:50-64); one gradient per draw with the current point's
    (logp, grad) cached on device.  ``sample()`` returns ``(theta, log p(theta))``.  A ``CudaModel`` with
    32 < dims <= 192 runs a kernel compiled at construction (``compile_log``: ptxas's report, ``""`` on every other
    engine)."""

    def __init__(self, model, epsilon: float, init=None, seed=None, *,
                 chains: Optional[int] = None, chain_offset: int = 0):
        super().__init__(model, init, seed, chains, chain_offset)
        self._epsilon = float(epsilon)
        if not self._epsilon > 0:
            raise ValueError(f"epsilon must be positive, got {epsilon}")
        self._prepare_wide("MALA")

    def _launch(self, n, rng, out, c0=0, cn=None, cache_valid=None):
        lib = L.lib()
        self._need_grad_cache()
        cn = self._C if cn is None else cn
        wp, wn = self._ws.get(lib.bk_mala_workspace_bytes(self._model.handle, self._C))
        L.check(lib.bk_mala_sample(
            self._model.handle, self._theta[c0:].data_ptr(), self._lp[c0:].data_ptr(),
            self._grad[c0:].data_ptr(), C.byref(self._cache_valid if cache_valid is None else cache_valid), cn, self._epsilon, n,
            C.byref(rng), C.byref(out), wp, wn, stream_ptr(self.device)))
