"""Device-side model plugins.

The reference's model boundary is the structural protocol of
bayes_kit/typing.py:15-42 (``dims()``, ``log_density(theta)``,
``log_density_gradient(theta)``, and for SMC ``log_prior`` / ``log_likelihood``),
called from the interpreter once per gradient.  Here a model is a *plugin
handle*: its parameters live on the device, it is registered with libbk_b200
(``bk_model_create``) and the samplers evaluate it inside their kernels -- no
Python callback per step.  The objects still implement the protocol (batched,
on device) so protocol-level user code keeps working.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L
from ._util import Workspace, compile_log, dtype_id, ptr, require_cuda, stream_ptr, to_dev


class DeviceModel:
    """Base of all plugins.  theta may be [D] (one point) or [C, D] (batched)."""

    _kind = None

    def __init__(self, dims, dtype, device):
        self.device = require_cuda(device)
        self.dtype = dtype
        self._dims = int(dims)
        self._handle = None
        self._keep = []          # tensors the handle points into
        self._ws = Workspace(self.device)
        self._model_ws = None

    def _register(self, **fields):
        d = L.ModelDesc()
        d.kind, d.dtype, d.dims = self._kind, dtype_id(self.dtype), self._dims
        d.sigma = float(fields.pop("sigma", 1.0))
        d.n_obs = int(fields.pop("n_obs", 0))
        for i, v in enumerate(fields.pop("scalars", ())):
            d.scalars[i] = float(v)
        for k, t in fields.items():
            if t is not None:
                self._keep.append(t)
                setattr(d, k, t.data_ptr())
        lib = L.lib()
        nbytes = lib.bk_model_workspace_bytes(C.byref(d))
        self._model_ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=self.device)
        h = L.u64(0)
        with torch.cuda.device(self.device):
            L.check(lib.bk_model_create(C.byref(d), self._model_ws.data_ptr(), self._model_ws.numel(),
                                        stream_ptr(self.device), C.byref(h)))
        self._handle = h.value

    def __del__(self):
        try:
            if self._handle is not None:
                L.lib().bk_model_destroy(self._handle)
        except Exception:
            pass

    @property
    def handle(self) -> int:
        return self._handle

    # ---- reference protocol (typing.py:15-27), batched -------------------------
    def dims(self) -> int:
        return self._dims

    def _eval(self, theta, want_grad, fast=False):
        th = to_dev(theta, self.dtype, self.device)
        single = th.dim() == 1
        th2 = th.reshape(1, -1) if single else th
        if th2.dim() != 2 or th2.shape[1] != self._dims:
            raise ValueError(f"theta must have shape [{self._dims}] or [C, {self._dims}]")
        Cn = th2.shape[0]
        lp = torch.empty(Cn, dtype=self.dtype, device=self.device)
        g = torch.empty_like(th2) if want_grad else None
        lib = L.lib()
        wp, wn = self._ws.get(lib.bk_model_eval_workspace_bytes(self._handle, Cn))
        with torch.cuda.device(self.device):
            fn = lib.bk_model_log_density_gradient_fast if fast else lib.bk_model_log_density_gradient
            L.check(fn(self._handle, th2.data_ptr(), Cn, lp.data_ptr(), ptr(g), wp, wn,
                       stream_ptr(self.device)))
        if single:
            return float(lp[0]), (g[0] if want_grad else None)
        return lp, g

    def log_density(self, theta):
        return self._eval(theta, False)[0]

    def log_density_gradient(self, theta, fast: bool = False):
        """``fast=True``: the reduced-precision (tensor-core) evaluation the samplers use
        for interior leapfrog steps, where the plugin has one."""
        return self._eval(theta, True, fast)


class IsoGauss(DeviceModel):
    """``log p = -0.5 |theta|^2 / sigma^2`` -- the D-dim generalisation of the
    reference's test model (test/models/std_normal.py:8-13)."""

    _kind = L.MODEL_ISO

    def __init__(self, dims, sigma=1.0, dtype=torch.float32, device="cuda"):
        super().__init__(dims, dtype, device)
        self.sigma = float(sigma)
        self._register(sigma=self.sigma)


StdNormal = IsoGauss


class DiagGauss(DeviceModel):
    """``log p = -0.5 sum prec_i (theta_i - mu_i)^2``."""

    _kind = L.MODEL_DIAG

    def __init__(self, mu, prec, dtype=torch.float32, device="cuda"):
        prec_np = np.asarray(prec.cpu() if isinstance(prec, torch.Tensor) else prec)
        super().__init__(prec_np.shape[0], dtype, device)
        self.mu = None if mu is None else to_dev(mu, dtype, self.device)
        self.prec = to_dev(prec, dtype, self.device)
        self._register(mu=self.mu, prec=self.prec)


class DensePrecGauss(DeviceModel):
    """``log p = -0.5 (theta-mu)^T P (theta-mu)`` with a dense symmetric
    precision (BASELINE config c2: P = A A^T / D + I)."""

    _kind = L.MODEL_DENSE

    def __init__(self, P, mu=None, dtype=torch.float32, device="cuda"):
        dev = require_cuda(device)
        Pt = to_dev(P, dtype, dev)
        if Pt.dim() != 2 or Pt.shape[0] != Pt.shape[1]:
            raise ValueError("P must be a square matrix")
        super().__init__(Pt.shape[0], dtype, dev)
        self.P = Pt
        self.mu = None if mu is None else to_dev(mu, dtype, self.device)
        self._register(P=self.P, mu=self.mu)


class GaussPriorLik(DeviceModel):
    """Tempering target for TemperedLikelihoodSMC (typing.py:37-42):
    ``log_prior = -0.5 sum p0 (theta-m0)^2``, ``log_likelihood = -0.5 sum pl (theta-mu)^2``."""

    _kind = L.MODEL_GPL

    def __init__(self, m0, p0, mu, pl, dtype=torch.float32, device="cuda"):
        dev = require_cuda(device)
        mu_t = to_dev(mu, dtype, dev)
        super().__init__(mu_t.shape[0], dtype, dev)
        self.mu, self.pl = mu_t, to_dev(pl, dtype, dev)
        self.m0, self.p0 = to_dev(m0, dtype, dev), to_dev(p0, dtype, dev)
        self._register(mu=self.mu, prec=self.pl, m0=self.m0, p0=self.p0)

    def _pl(self, theta, which):
        th = to_dev(theta, self.dtype, self.device)
        single = th.dim() == 1
        th2 = th.reshape(1, -1) if single else th
        out = torch.empty(th2.shape[0], dtype=self.dtype, device=self.device)
        args = (out.data_ptr(), None) if which == "prior" else (None, out.data_ptr())
        with torch.cuda.device(self.device):
            L.check(L.lib().bk_model_log_prior_likelihood(self._handle, th2.data_ptr(), th2.shape[0],
                                                          *args, stream_ptr(self.device)))
        return float(out[0]) if single else out

    def log_prior(self, theta):
        return self._pl(theta, "prior")

    def log_likelihood(self, theta):
        return self._pl(theta, "lik")


class Binomial(DeviceModel):
    """Beta-binomial on the logit scale -- the reference's own test target
    (test/models/binomial.py:11-74): ``theta = logit(p)``, ``x ~ Binomial(N, p)``,
    ``p ~ Beta(alpha, beta)`` with the logit Jacobian; ``log_prior`` / ``log_likelihood`` for the SMC
    (binomial.py:44-54), analytic gradient (the reference differentiates numerically)."""

    _kind = L.MODEL_BINOM

    def __init__(self, alpha, beta, x, N, dtype=torch.float32, device="cuda"):
        import math
        super().__init__(1, dtype, device)
        self.alpha, self.beta, self.x, self.N = float(alpha), float(beta), int(x), int(N)
        lch = math.lgamma(N + 1) - math.lgamma(x + 1) - math.lgamma(N - x + 1)
        lbe = math.lgamma(alpha) + math.lgamma(beta) - math.lgamma(alpha + beta)
        self._register(scalars=(alpha, beta, x, N, lch, lbe))

    _pl = GaussPriorLik._pl
    log_prior = GaussPriorLik.log_prior
    log_likelihood = GaussPriorLik.log_likelihood

    def constrain_draws(self, draws):      # binomial.py:67-68
        return torch.sigmoid(draws)

    def posterior_mean(self) -> float:     # binomial.py:70-74
        a, b = self.alpha + self.x, self.beta + self.N - self.x
        return a / (a + b)

    def posterior_variance(self) -> float:
        a, b = self.alpha + self.x, self.beta + self.N - self.x
        return a * b / ((a + b) ** 2 * (a + b + 1))


class HierLogReg(DeviceModel):
    """Hierarchical logistic regression (BASELINE config c3; density in DESIGN.md)."""

    _kind = L.MODEL_HLR

    def __init__(self, X, y, dtype=torch.float32, device="cuda"):
        dev = require_cuda(device)
        Xt = to_dev(X, dtype, dev)
        super().__init__(Xt.shape[1] + 2, dtype, dev)
        self.X, self.y = Xt, to_dev(y, dtype, dev)
        self._register(X=self.X, y=self.y, n_obs=Xt.shape[0])


_NVRTC_LOADED = False


def _load_nvrtc() -> None:
    """Make ``libnvrtc.so.12`` loadable by soname for the library's ``dlopen``: the system copy when the
    loader finds one, else the copy bundled with torch (nvidia-cuda-nvrtc), loaded ``RTLD_GLOBAL``."""
    global _NVRTC_LOADED
    if _NVRTC_LOADED:
        return
    try:
        C.CDLL("libnvrtc.so.12", mode=C.RTLD_GLOBAL)
    except OSError:
        import glob
        import os
        import sys
        for base in sys.path:
            for cand in glob.glob(os.path.join(base, "nvidia", "cuda_nvrtc", "lib", "libnvrtc.so.12")):
                try:
                    C.CDLL(cand, mode=C.RTLD_GLOBAL)
                    _NVRTC_LOADED = True
                    return
                except OSError:
                    pass
        return          # bk_model_create_cuda reports BK_E_UNSUPPORTED
    _NVRTC_LOADED = True


class CudaModel(DeviceModel):
    """A model written by the user as one CUDA C++ function, compiled at run time (NVRTC) for the GPU::

        __device__ bk_real log_density_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);

    It returns ``log p(theta)`` and writes the gradient into ``grad[0 .. BK_DIMS)``; ``bk_real`` is the model's
    dtype and ``BK_DIMS == dims`` a compile-time constant.  Helper functions, structs and constants may precede
    it; no header can be included (math builtins need none).  ``params``: the model's data and
    hyper-parameters as one flat array, passed to the function on the device.

    Every sampler except ``TemperedLikelihoodSMC`` accepts it; for the SMC, write the log prior and the log
    likelihood separately as a ``CudaPriorLikModel``.  ``HMCDiag``, ``MALA``, the random-walk
    ``Metropolis`` / ``MetropolisHastings``, ``DrGhmcDiag`` and the ``Stretcher`` run one fused kernel per call
    (one thread per chain or walker, state in registers) for ``dims <= 32``, the generic engines above; the
    kernels of ``DrGhmcDiag`` and the ``Stretcher`` are compiled when the sampler is constructed.  A compile
    error raises ``ValueError`` with NVRTC's log; ``compile_log`` holds the log of a successful compile, with
    the registers and spills of every kernel."""

    _kind = L.MODEL_USER
    _create = "bk_model_create_cuda"

    def __init__(self, source: str, dims: int, params=None, dtype=torch.float32, device="cuda"):
        if not isinstance(source, str):
            raise TypeError("source must be a str of CUDA C++")
        if isinstance(dims, bool) or not isinstance(dims, (int, np.integer)):
            raise TypeError(f"dims must be an int, not {type(dims)}")
        super().__init__(dims, dtype, device)
        self.source = source
        self.params = None
        if params is not None:
            self.params = to_dev(params, dtype, self.device).reshape(-1)
            if self.params.numel() == 0:
                self.params = None
        n_params = 0 if self.params is None else self.params.numel()
        _load_nvrtc()
        h = L.u64(0)
        create = getattr(L.lib(), self._create)
        self.compile_log = compile_log(
            lambda log, n: create(source.encode(), self._dims, dtype_id(dtype), ptr(self.params), n_params,
                                  C.byref(h), log, n),
            f"{type(self).__name__}: NVRTC compilation failed:\n", self.device)
        self._handle = h.value


class CudaPriorLikModel(CudaModel):
    """A model written by the user as a log prior and a log likelihood, compiled at run time (NVRTC), for
    ``TemperedLikelihoodSMC`` (the reference's ``LogPriorLikelihoodModel``, typing.py:37-42)::

        __device__ bk_real log_prior_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);
        __device__ bk_real log_likelihood_gradient(const bk_real* theta, bk_real* grad, const bk_real* params);

    Each returns its log term and writes that term's gradient into ``grad[0 .. BK_DIMS)``; ``bk_real``,
    ``BK_DIMS``, ``params`` and helper code are as for ``CudaModel``.  ``dims <= 256`` (the SMC's limit;
    ``ValueError`` above).  The library derives ``log_density_gradient`` = likelihood + prior from the pair, so the
    same object also runs on every MCMC sampler, targeting the posterior.  The SMC moves its particles with one
    thread per particle (RW / MALA / HMC kernels, sharded or not).  ``log_prior`` / ``log_likelihood`` are batched
    on the device like ``GaussPriorLik``'s."""

    _create = "bk_model_create_cuda_prior_lik"

    _pl = GaussPriorLik._pl
    log_prior = GaussPriorLik.log_prior
    log_likelihood = GaussPriorLik.log_likelihood


def require_plugin(model) -> DeviceModel:
    if not isinstance(model, DeviceModel):
        raise TypeError(
            "bayes_kit_b200 samplers evaluate the model inside CUDA kernels: `model` must be a "
            "registered device plugin (bayes_kit_b200.models.IsoGauss / DiagGauss / DensePrecGauss / "
            "HierLogReg / GaussPriorLik / Binomial, or your own CUDA source as CudaModel / CudaPriorLikModel), not an arbitrary Python object. Python callbacks cannot "
            f"run per step on the device and there is no CPU fallback (got {type(model).__name__}).")
    return model
