"""Metropolis / MetropolisHastings (reference: bayes_kit/metropolis.py).

The reference takes arbitrary Python callables ``proposal_fn(theta)`` and
``transition_lp_fn(to, from)`` (metropolis.py:79-88).  Python callbacks cannot
run per step on the device and there is no CPU fallback, so the proposal is a
*device proposal descriptor*: the built-in ``GaussianRW(scale)`` -- the family
the reference's tests and SMC kernel use (test_metropolis.py:114,
smc.py:79-89) -- or a ``CudaProposal``, the proposal and its transition density
written by the user in CUDA C++ and compiled at run time.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from ._sampler import ChainSampler
from ._util import compile_log, dtype_id, ptr, require_cuda, stream_ptr, to_dev


def metropolis_accept_test(lp_proposal: float, lp_current: float, rng) -> bool:
    """metropolis.py:12-38 (host scalar form, strict ``<``; ``log(0) = -inf``
    always accepts)."""
    u = rng.uniform()
    log_u = math.log(u) if u > 0 else -math.inf
    return log_u < lp_proposal - lp_current


def metropolis_hastings_accept_test(lp_proposal: float, lp_current: float,
                                    lp_forward_transition: float, lp_reverse_transition: float,
                                    rng) -> bool:
    """metropolis.py:41-76."""
    u = rng.uniform()
    log_u = math.log(u) if u > 0 else -math.inf
    return log_u < (lp_proposal - lp_current) + (lp_reverse_transition - lp_forward_transition)


class GaussianRW:
    """Symmetric Gaussian random-walk proposal ``theta' = theta + scale * z``."""

    def __init__(self, scale: float):
        self.scale = float(scale)
        if not self.scale > 0:
            raise ValueError(f"scale must be positive, got {scale}")

    def transition_lp(self, to, frm):  # marker, evaluated on device
        raise TypeError("GaussianRW.transition_lp is a device-side descriptor; pass it to "
                        "MetropolisHastings, do not call it")


class CudaProposal:
    """A proposal written by the user in CUDA C++, compiled at run time (NVRTC) for the GPU::

        __device__ void propose(const bk_real* theta, bk_real* proposal, const bk_real* z, const bk_real* u,
                                const bk_real* params);
        __device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* params);

    ``propose`` writes theta' into ``proposal[0 .. BK_DIMS)`` from ``z`` (``normals`` standard normals, default
    ``dims``) and ``u`` (``uniforms`` uniforms in (0, 1)) that the library draws for every chain and draw;
    ``transition_log_density`` returns ``log q(to | from)`` up to a constant and is needed only with
    ``transition=True`` (``MetropolisHastings``).  ``bk_real``, ``BK_DIMS``, ``params`` and helper code are as for
    ``CudaModel``; the source is compiled inside a namespace of its own, so its helpers may share names with the
    model's.  Pass the object as ``proposal_fn`` and its ``transition_lp`` as ``transition_lp_fn``.  With a
    ``CudaModel`` of ``dims <= 32`` (and ``normals <= 32``) the sampler runs one fused kernel per call, compiled at
    construction; otherwise three launches per draw (proposal, model, accept test).  A compile error raises
    ``ValueError`` with NVRTC's log; ``compile_log`` holds the log of a successful compile.

    With ``gradient=True`` the proposal also reads the gradient of the sampler's model (MALA, preconditioned MALA,
    the Barker proposal, any drift-plus-noise move)::

        __device__ void propose(const bk_real* theta, const bk_real* grad, bk_real* proposal, const bk_real* z,
                                const bk_real* u, const bk_real* params);
        __device__ bk_real transition_log_density(const bk_real* to, const bk_real* from, const bk_real* grad_from,
                                                  const bk_real* params);

    ``grad`` is ``grad log p(theta)`` and ``grad_from`` is ``grad log p(from)``; the Hastings term is
    ``transition_log_density(theta, q, grad log p(q)) - transition_log_density(q, theta, grad log p(theta))``.  The
    fused kernel keeps the gradient in registers; every other model runs four launches per draw (proposal, the
    model's log density and gradient, the Hastings term, accept test), three without a Hastings term.  The SMC's
    ``proposal_kernel`` does not take a gradient proposal."""

    def __init__(self, source: str, dims: int, params=None, normals=None, uniforms: int = 0, transition: bool = True,
                 dtype=torch.float32, device="cuda", gradient: bool = False):
        from .models import _load_nvrtc
        if not isinstance(source, str):
            raise TypeError("source must be a str of CUDA C++")
        for name, v in (("dims", dims), ("normals", dims if normals is None else normals), ("uniforms", uniforms)):
            if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
                raise TypeError(f"{name} must be an int, not {type(v)}")
        self._handle = None
        self.device = require_cuda(device)
        self.dtype = dtype
        self.source = source
        self.dims = int(dims)
        self.normals = self.dims if normals is None else int(normals)
        self.uniforms = int(uniforms)
        self.transition = bool(transition)
        self.gradient = bool(gradient)
        self.params = None
        if params is not None:
            self.params = to_dev(params, dtype, self.device).reshape(-1)
            if self.params.numel() == 0:
                self.params = None
        n_params = 0 if self.params is None else self.params.numel()
        _load_nvrtc()
        h = L.u64(0)
        create = L.lib().bk_proposal_create_cuda_grad if self.gradient else L.lib().bk_proposal_create_cuda
        self.compile_log = compile_log(
            lambda log, n: create(source.encode(), self.dims, dtype_id(dtype), ptr(self.params), n_params,
                                  self.normals, self.uniforms, int(self.transition), C.byref(h), log, n),
            "CudaProposal: NVRTC compilation failed:\n", self.device)
        self._handle = h.value

    @property
    def handle(self) -> int:
        return self._handle

    def transition_lp(self, to, frm):  # marker, evaluated on device
        raise TypeError("CudaProposal.transition_lp is a device-side descriptor; pass it to MetropolisHastings, "
                        "do not call it")

    def __del__(self):
        try:
            if self._handle is not None:
                L.lib().bk_proposal_destroy(self._handle)
        except Exception:
            pass


def _require_proposal(proposal_fn):
    if not isinstance(proposal_fn, (GaussianRW, CudaProposal)):
        raise TypeError(
            "proposal_fn must be a device proposal descriptor (bayes_kit_b200.GaussianRW(scale) or a "
            "bayes_kit_b200.CudaProposal written in CUDA C++): arbitrary Python callables cannot run per step on the "
            "GPU and there is no CPU fallback")
    return proposal_fn


class MetropolisHastings(ChainSampler):
    """``MetropolisHastings(model, proposal_fn, transition_lp_fn, *, init=None,
    seed=None)`` (metropolis.py:80-99).  ``transition_lp_fn`` must be the
    proposal's own ``transition_lp`` (the Hastings terms are evaluated on
    device; they cancel exactly for a symmetric proposal).  With ``GaussianRW`` and a ``CudaModel`` with
    32 < dims <= 192 the sampler runs a kernel compiled at construction (``compile_log``: ptxas's report, ``""`` on
    every other engine)."""

    _hastings = 1

    def __init__(self, model, proposal_fn, transition_lp_fn, *, init=None, seed=None,
                 chains: Optional[int] = None, chain_offset: int = 0):
        prop = _require_proposal(proposal_fn)
        if self._hastings and isinstance(prop, CudaProposal) and not prop.transition:
            raise TypeError("MetropolisHastings needs the proposal's transition density: create the CudaProposal "
                            "with transition=True (and define transition_log_density), or use Metropolis")
        if self._hastings and getattr(transition_lp_fn, "__self__", None) is not prop:
            raise TypeError("transition_lp_fn must be proposal_fn.transition_lp (device descriptor)")
        super().__init__(model, init, seed, chains, chain_offset)
        self._proposal_fn = prop
        self._transition_lp_fn = transition_lp_fn
        if isinstance(prop, CudaProposal):
            if prop.dims != self._dim or prop.dtype != self.dtype:
                raise ValueError(f"the proposal (dims {prop.dims}, {prop.dtype}) does not match the model "
                                 f"(dims {self._dim}, {self.dtype})")
            self._n_normal, self._n_uniform = prop.normals, 1 + prop.uniforms
            # gradient proposals, three-launch path: the library caches grad log p(theta) in the workspace, for the
            # rows of the last call; a call on other rows (sample_host's chunks) re-evaluates it
            self._ws_grad_rows = None
            # compile the fused kernel now, not in the first sample(); its log, or "" (three launches)
            self.compile_log = compile_log(
                lambda log, n: L.lib().bk_mh_cuda_prepare(self._model.handle, prop.handle, log, n),
                "MetropolisHastings: NVRTC compilation of the model with the proposal failed:\n", self.device)
        else:
            self._prepare_wide(type(self).__name__)

    def _fuses_extras(self) -> bool:
        return not isinstance(self._proposal_fn, CudaProposal) and super()._fuses_extras()

    def _launch(self, n, rng, out, c0=0, cn=None, cache_valid=None):
        lib = L.lib()
        cn = self._C if cn is None else cn
        valid = self._cache_valid if cache_valid is None else cache_valid
        cv = C.byref(valid)
        prop = self._proposal_fn
        if isinstance(prop, CudaProposal):
            wp, wn = self._ws.get(lib.bk_mh_cuda_workspace_bytes(self._model.handle, prop.handle, self._C))
            if prop.gradient:
                if self._ws_grad_rows != (c0, cn):
                    valid.value = 0
                self._ws_grad_rows = (c0, cn)
            L.check(lib.bk_mh_cuda_sample(
                self._model.handle, prop.handle, self._theta[c0:].data_ptr(), self._lp[c0:].data_ptr(), cv, cn,
                self._hastings, n, C.byref(rng), C.byref(out), wp, wn, stream_ptr(self.device)))
            return
        wp, wn = self._ws.get(lib.bk_mh_rw_workspace_bytes(self._model.handle, self._C))
        L.check(lib.bk_mh_rw_sample(
            self._model.handle, self._theta[c0:].data_ptr(), self._lp[c0:].data_ptr(),
            cv, cn, prop.scale, self._hastings, n,
            C.byref(rng), C.byref(out), wp, wn, stream_ptr(self.device)))


class Metropolis(MetropolisHastings):
    """``Metropolis(model, proposal_fn, *, init=None, seed=None)``
    (metropolis.py:138-155): symmetric proposal, no Hastings term."""

    _hastings = 0

    def __init__(self, model, proposal_fn, *, init=None, seed=None, chains: Optional[int] = None,
                 chain_offset: int = 0):
        super().__init__(model, proposal_fn, None, init=init, seed=seed, chains=chains,
                         chain_offset=chain_offset)
