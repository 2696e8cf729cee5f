"""DrGhmcDiag -- delayed-rejection generalized HMC (reference: bayes_kit/drghmc.py;
Modi, Barnett, Carpenter 2023)."""
from __future__ import annotations

import ctypes as C
from collections.abc import Sequence
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from ._sampler import ChainSampler, _is_empty_init
from ._util import compile_log, ptr, stream_ptr, to_dev
from .models import CudaModel


class DrGhmcDiag(ChainSampler):
    """``DrGhmcDiag(model, max_proposals, leapfrog_step_sizes, leapfrog_step_counts,
    damping, metric_diag=None, init=None, seed=None, prob_retry=True)``
    (drghmc.py:37-48), same argument validation and error messages
    (drghmc.py:85-207).

    Per draw (drghmc.py:348-389): partial momentum refresh
    ``rho <- rho sqrt(1-damping) + sqrt(damping) z``, up to ``max_proposals``
    leapfrog proposals with probabilistic retry, ghost-proposal Hastings terms
    (drghmc.py:391-446), unconditional momentum flip.  ``sample()`` returns
    ``(theta, joint_logp)``.  Every chain follows its own data-dependent
    proposal schedule inside one fused kernel (explicit recursion on the
    proposal index instead of Python recursion) on iso / diagonal Gaussians
    and on a ``CudaModel`` / ``CudaPriorLikModel`` with ``dims <= 32``; the
    latter's kernel is compiled from the model's source at construction
    (``compile_log``: ptxas's report, ``""`` on every other engine; a compile
    error raises ``ValueError`` with NVRTC's log).  Every other model runs
    the lockstep engine.
    """

    def __init__(self, model, max_proposals, leapfrog_step_sizes, leapfrog_step_counts, damping,
                 metric_diag=None, init=None, seed=None, prob_retry: bool = True, *,
                 chains: Optional[int] = None, chain_offset: int = 0):
        self._max_proposals = max_proposals
        self._leapfrog_step_sizes = leapfrog_step_sizes
        self._leapfrog_step_counts = leapfrog_step_counts
        self._damping = damping
        self._prob_retry = prob_retry
        self._validate_arguments()
        super().__init__(model, init, seed, chains, chain_offset)
        self._n_uniform = 2 * int(max_proposals)
        if metric_diag is None:
            self._metric = None
        else:
            m = to_dev(metric_diag, self.dtype, self.device).reshape(-1)
            if m.numel() == 1 and self._dim > 1:
                m = m.expand(self._dim).contiguous()
            if m.numel() != self._dim:
                raise ValueError(f"metric_diag must have {self._dim} entries")
            self._metric = m
        # rho0 ~ N(0, I) (drghmc.py:77): device Philox keyed by the global chain id, like theta0
        self._rho = self._philox_normal(self._C, 0xFFFFFFFE)
        self._sizes = (C.c_double * int(max_proposals))(*[float(s) for s in leapfrog_step_sizes])
        self._counts = (C.c_int32 * int(max_proposals))(*[int(c) for c in leapfrog_step_counts])
        self.last_n_uniform = None
        self.compile_log = ""
        if isinstance(self._model, CudaModel):
            # compile the fused kernel now, not in the first sample(); its log, or "" (lockstep engine)
            self.compile_log = compile_log(
                lambda log, n: L.lib().bk_drghmc_cuda_prepare(self._model.handle, log, n),
                "DrGhmcDiag: NVRTC compilation of the model's DrGHMC kernel failed:\n", self.device)

    @property
    def rho(self) -> torch.Tensor:
        return self._rho[0] if self._single else self._rho

    def set_momentum(self, rho) -> None:
        """Overwrite the persistent momentum (parity tests feed the reference's rho0)."""
        self._rho = to_dev(rho, self.dtype, self.device).reshape(self._C, self._dim).clone()

    # ---- argument validation: types and messages of drghmc.py:85-207 ---------------
    def _validate_arguments(self) -> None:
        k = self._max_proposals
        if not isinstance(k, int):
            raise TypeError(f"max_proposals must be an int, not {type(k)}")
        if not (k >= 1):
            raise ValueError(f"max_proposals must be greater than or equal to 1, not {k}")
        self._validate_seq(self._leapfrog_step_sizes, "leapfrog_step_sizes", "step size", float,
                           "leapfrog step size")
        self._validate_seq(self._leapfrog_step_counts, "leapfrog_step_counts", "step count", int,
                           "number of leapfrog steps")
        d = self._damping
        if not isinstance(d, float):
            raise TypeError(f"damping must be of type float, but found type {type(d)}")
        if not 0 < d <= 1:
            raise ValueError(f"damping must be within (0, 1], but found damping of {d}")

    def _validate_seq(self, seq, name, item, typ, what) -> None:
        if not isinstance(seq, Sequence):
            raise TypeError(f"{name} must be an instance of type sequence, but found type {type(seq)}")
        if len(seq) != self._max_proposals:
            raise ValueError(
                f"{name} must be a sequence of length {self._max_proposals}, so that each proposal "
                f"has its own specified {what}, but instead found length of {len(seq)}")
        for idx, v in enumerate(seq):
            if not isinstance(v, typ):
                raise TypeError(f"each {item} in {name} must be of type {typ.__name__}, but found "
                                f"{item} of type {type(v)} at index {idx}")
            if not v > 0:
                raise ValueError(f"each {item} in {name} must be positive, but found {item} of {v} "
                                 f"at index {idx}")

    def _launch(self, n, rng, out, c0=0, cn=None, cache_valid=None):
        """``c0, cn``: a chunk of chains (``sample_host`` pipelines chunks over PCIe); the persistent momentum of the
        chunk's chains stays on the device, exactly as ``_rho`` is internal state upstream (drghmc.py:77,388)."""
        lib = L.lib()
        cn = self._C if cn is None else cn
        if c0 == 0:
            self._used = torch.empty(n, self._C, dtype=torch.int32, device=self.device)
        used = self._used if cn == self._C else torch.empty(n, cn, dtype=torch.int32, device=self.device)
        wp, wn = self._ws.get(lib.bk_drghmc_workspace_bytes(self._model.handle, cn, self._max_proposals))
        L.check(lib.bk_drghmc_sample(
            self._model.handle, self._theta[c0:].data_ptr(), self._rho[c0:].data_ptr(), cn,
            self._max_proposals, self._sizes, self._counts, float(self._damping),
            1 if self._prob_retry else 0, ptr(self._metric), n, C.byref(rng), C.byref(out),
            used.data_ptr(), wp, wn, stream_ptr(self.device)))
        if cn != self._C:
            self._used[:, c0:c0 + cn].copy_(used)
        self.last_n_uniform = self._used[:, 0] if self._single else self._used
