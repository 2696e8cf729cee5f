"""TemperedLikelihoodSMC (reference: bayes_kit/smc.py).

All M particles move, reweight and resample on device, one temperature per
``transition(n)``: a fused move + log-weight kernel (random-walk Metropolis as in
the reference, or a MALA / HMC transition -- the TODO of smc.py:78), a single-pass
fixed-point scan and a resolve kernel -- three launches per temperature.

Particles shard across the GPUs of a box (one process per GPU).  No host-side
collective runs per temperature and no particle array is exchanged: the ranks post
three small messages per step into each other's mailboxes (local max of the
log-weights, local weight mass, "indices final"), store the resample indices of the
offspring they resolve straight into the owner's index array, and the next move
reads the selected rows from their owners over NVLink peer memory (peer.py, bk.h).

The model is a built-in plugin with a log_prior / log_likelihood split (GaussPriorLik,
Binomial: lane-grouped move kernel) or the user's own CUDA source as a
CudaPriorLikModel (runtime-compiled move kernel, one thread per particle, same
random streams, resampling and cross-rank messages).  On a CudaPriorLikModel the
move may also be one Metropolis(-Hastings) step of a user-written CudaProposal
(``proposal_kernel``), compiled together with the model into one kernel.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterator, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from . import dist as D_
from . import peer as P_
from ._util import compile_log, make_rng, resolve_seed, stream_ptr, to_dev
from .metropolis import CudaProposal
from .models import Binomial, CudaPriorLikModel, GaussPriorLik, require_plugin


class _Kernel:
    kind = L.SMC_KERNEL_RW
    steps = 0

    def __init__(self, scale: float, what: str = "scale"):
        self.scale = float(scale)
        if not self.scale > 0:
            raise ValueError(f"{what} must be positive, got {scale}")

    def desc(self) -> L.SmcKernel:
        return L.SmcKernel(self.kind, self.steps, self.scale)

    def stream_widths(self, D: int):
        """(normals, uniforms) per particle of the injected streams."""
        return D, 1


class RWMetropolisKernel(_Kernel):
    """Device descriptor returned by ``metropolis_kernel(scale)``: one
    random-walk Metropolis move ``theta* = normal(loc=theta, scale)`` accepted
    iff ``log(u) < lp(theta*) - lp(theta)`` (smc.py:79-89)."""


class MALAKernel(_Kernel):
    """One MALA transition (mala.py:40-66) on the tempered density ``lp_t = ll * t + prior``."""
    kind = L.SMC_KERNEL_MALA

    def __init__(self, epsilon: float):
        super().__init__(epsilon, "epsilon")


class HMCKernel(_Kernel):
    """One HMCDiag transition (hmc.py:40-63, identity metric) on the tempered density."""
    kind = L.SMC_KERNEL_HMC

    def __init__(self, stepsize: float, steps: int):
        super().__init__(stepsize, "stepsize")
        self.steps = int(steps)
        if self.steps < 0:
            raise ValueError(f"steps must be >= 0, got {steps}")


class ProposalKernel(_Kernel):
    """One Metropolis(-Hastings) step of a user-written ``CudaProposal`` on the tempered density
    ``lp_t = ll * t + prior``: ``theta* = propose(theta, z, u)``, accepted iff ``log(u_acc) < lp_t(theta*) -
    lp_t(theta)`` plus, for a proposal created with ``transition=True``, ``log q(theta | theta*) - log q(theta* |
    theta)`` (the reference's ``kernel`` argument with any Markov kernel, smc.py:54-57).  Runs on a
    ``CudaPriorLikModel`` of the proposal's dims and dtype, compiled together with it into one kernel."""
    kind = L.SMC_KERNEL_PROPOSAL

    def __init__(self, proposal):
        if not isinstance(proposal, CudaProposal):
            raise TypeError("proposal_kernel needs a bayes_kit_b200.CudaProposal written in CUDA C++ "
                            f"(got {type(proposal).__name__})")
        self.proposal = proposal          # keeps the handle alive as long as the kernel

    def desc(self) -> L.SmcKernel:
        return L.SmcKernel(self.kind, 0, 0.0, self.proposal.handle)

    def stream_widths(self, D: int):
        return self.proposal.normals, 1 + self.proposal.uniforms


def metropolis_kernel(scale: float) -> RWMetropolisKernel:
    return RWMetropolisKernel(scale)


def mala_kernel(epsilon: float) -> MALAKernel:
    """MCMC-kernel plug-in for the SMC (the TODO at smc.py:78)."""
    return MALAKernel(epsilon)


def hmc_kernel(stepsize: float, steps: int) -> HMCKernel:
    """MCMC-kernel plug-in for the SMC (the TODO at smc.py:78)."""
    return HMCKernel(stepsize, steps)


def proposal_kernel(proposal: CudaProposal) -> ProposalKernel:
    """MCMC-kernel plug-in for the SMC: one Metropolis(-Hastings) step of a user-written ``CudaProposal``."""
    return ProposalKernel(proposal)


class TemperedLikelihoodSMC:
    """``TemperedLikelihoodSMC(model, M, N, sample_initial, kernel)`` (smc.py:13-27).

    * ``model``: a plugin with ``log_prior`` / ``log_likelihood``: ``GaussPriorLik``, ``Binomial``, or the user's
      own CUDA source as a ``CudaPriorLikModel`` (dims <= 256).
    * ``sample_initial``: the reference's callable ``m -> theta0[m]`` (evaluated
      once per particle on the host, as smc.py:23 does), or directly an [M, D]
      array / tensor.
    * ``kernel``: ``metropolis_kernel(scale)`` (the reference's), ``mala_kernel(eps)``, ``hmc_kernel(eps, L)``,
      or, on a ``CudaPriorLikModel``, ``proposal_kernel(CudaProposal(...))``.  The fused program of the model and
      the proposal is compiled at construction (``compile_log``: ptxas's report, else "").
    * ``resample``: ``"multinomial"`` (reference semantics: no max-shift, legacy
      ``np.random.choice`` indices) or ``"systematic"`` (log-sum-exp normalised,
      stratified points, exact fixed-point CDF: the indices do not depend on how the
      particles are sharded; north_star item 2).
    * ``ess_threshold``: None (the reference: resample at every temperature,
      smc.py:60) or a fraction in (0, 1]: resample only when the importance-weight
      ESS drops below ``ess_threshold * M``, carrying the log-weights otherwise
      (``log_weights``, ``resampled``); the decision is taken on device.
    With torch.distributed initialised (or ``group=`` given), M is the GLOBAL particle
    count and each rank owns a contiguous slice.
    """

    def __init__(self, model, M: int, N: int, sample_initial, kernel, *, resample: str = "multinomial",
                 ess_threshold: Optional[float] = None, seed=None, group=None):
        self._model = require_plugin(model)
        if not isinstance(self._model, (GaussPriorLik, Binomial, CudaPriorLikModel)):
            raise TypeError("TemperedLikelihoodSMC needs a model plugin with log_prior/log_likelihood "
                            "(bayes_kit_b200.models.GaussPriorLik / Binomial / CudaPriorLikModel)")
        if not isinstance(kernel, _Kernel):
            raise TypeError("kernel must be bayes_kit_b200.metropolis_kernel(scale) (or mala_kernel / hmc_kernel / "
                            "proposal_kernel): arbitrary Python kernels cannot run per particle on the GPU and there is "
                            "no CPU fallback")
        self.compile_log = ""
        if isinstance(kernel, ProposalKernel):
            self._prepare(kernel.proposal)
        if resample not in ("multinomial", "systematic"):
            raise ValueError("resample must be 'multinomial' or 'systematic'")
        if ess_threshold is not None and not 0 < ess_threshold <= 1:
            raise ValueError(f"ess_threshold must be in (0, 1], got {ess_threshold}")
        if ess_threshold is not None and resample != "systematic":
            raise ValueError("ess_threshold needs resample='systematic'")
        self.ess_threshold = ess_threshold      # None: resample at every temperature (smc.py:60)
        self.M, self.N = int(M), int(N)
        self.kernel = kernel
        self.resample = resample
        self._mode = L.RESAMPLE_MULTINOMIAL if resample == "multinomial" else L.RESAMPLE_SYSTEMATIC
        self.device, self.dtype = self._model.device, self._model.dtype
        self._dt = L.BK_F32 if self.dtype == torch.float32 else L.BK_F64
        self._group = group
        self._rank, self._world = P_.rank_world(group)
        if self._world > L.SMC_MAX_WORLD:
            raise ValueError(f"at most {L.SMC_MAX_WORLD} ranks")
        if self.M < self._world:
            raise ValueError("need at least one particle per rank")
        self._seed = D_.shared_seed(resolve_seed(seed), None if isinstance(group, P_.FakeRank) else group,
                                    self.device) if seed is None else resolve_seed(seed)
        self._lo, self._hi = D_.shard_range(self.M, self._rank, self._world)
        if callable(sample_initial):
            th = np.array([np.asarray(sample_initial(m), dtype=np.float64)
                           for m in range(self._lo, self._hi)])
            th = th.reshape(self._hi - self._lo, -1)
        else:
            th = sample_initial
            if th.shape[0] == self.M and self._world > 1:
                th = th[self._lo:self._hi]
        self._src_local = to_dev(th, self.dtype, self.device).clone()   # particles the next move starts from
        self._pending = False   # True: the current particles are rows idx[m] of the step's arrays (not materialised)
        self.D = self._src_local.shape[1]
        if self.D != self._model.dims():
            raise ValueError("sample_initial returned the wrong dimension")
        if self._src_local.shape[0] != self._hi - self._lo:
            raise ValueError("sample_initial returned the wrong number of particles")
        # ---- peer-addressable state: two particle arrays, log-weights, indices, mailbox ----------
        es = 4 if self.dtype == torch.float32 else 8
        n_max = -(-self.M // self._world)
        key = f"smc{id(self) if not isinstance(group, P_.FakeRank) else ''}:{self.M}:{self.D}:{es}"
        self._mem = P_.PeerRegion(key, {"p0": n_max * self.D * es, "p1": n_max * self.D * es, "l0": n_max * 2 * es,
                                        "l1": n_max * 2 * es, "logw": n_max * es,
                                        "idx": n_max * 8, "mail": L.SMC_MAILBOX_BYTES}, self.device, group)
        nl = self._hi - self._lo
        self._parts = [self._mem.tensor("p0", self.dtype, (nl, self.D)), self._mem.tensor("p1", self.dtype, (nl, self.D))]
        self._logw = self._mem.tensor("logw", self.dtype, (nl,))
        self._idx = self._mem.tensor("idx", torch.int64, (nl,))
        self._mail = self._mem.tensor("mail", torch.int64, (L.SMC_MAILBOX_BYTES // 8,))
        self._ws = torch.zeros(int(L.lib().bk_smc_shard_workspace_bytes(self.M, self._world, self._mode)),
                               dtype=torch.uint8, device=self.device)
        self._stats = torch.zeros(self.N + 1, 4, dtype=torch.float64, device=self.device)
        self._epoch = 0
        self._steps_taken = []
        self._shard = None
        self.last_accept = None

    def _prepare(self, prop: CudaProposal) -> None:
        """Check (model, proposal) and compile their fused program now, not in the first move."""
        if not isinstance(self._model, CudaPriorLikModel):
            raise NotImplementedError("proposal_kernel runs on a CudaPriorLikModel only: restate the built-in "
                                      f"{type(self._model).__name__} as a CudaPriorLikModel")
        if prop.dims != self._model.dims() or prop.dtype != self._model.dtype:
            raise ValueError(f"the proposal (dims {prop.dims}, {prop.dtype}) does not match the model "
                             f"(dims {self._model.dims()}, {self._model.dtype})")
        self.compile_log = compile_log(
            lambda log, n: L.lib().bk_smc_cuda_prepare(self._model.handle, prop.handle, log, n),
            "TemperedLikelihoodSMC: NVRTC compilation of the model with the proposal failed:\n", self._model.device)

    # ---- plumbing --------------------------------------------------------------------
    def _sh(self) -> L.SmcShard:
        if self._shard is None:
            s = L.SmcShard()
            s.rank, s.world, s.M = self._rank, self._world, self.M
            for name, field in (("p0", s.particles[0]), ("p1", s.particles[1]), ("l0", s.llpr[0]), ("l1", s.llpr[1]),
                                ("logw", s.logw), ("idx", s.idx),
                                ("mail", s.mailbox)):
                for r, p in enumerate(self._mem.ptrs(name)):
                    field[r] = p
            self._shard = s
        self._shard.epoch = self._epoch
        return self._shard

    def _check(self) -> None:
        """Raise if a kernel flagged the mailbox (synchronises)."""
        err = int(self._mail[0].item())
        if err == 1:
            raise L.BkError("TemperedLikelihoodSMC: a rank did not arrive within 20 s (dead peer?); the particles are invalid")
        if err == 2:
            raise FloatingPointError("TemperedLikelihoodSMC: every importance weight vanished")

    # ---- reference surface -----------------------------------------------------------
    @property
    def thetas(self) -> torch.Tensor:
        """Current particles [M_local, D] (smc.py:23,60).  The resampling gather
        ``thetas[idxs]`` (smc.py:75) is normally folded into the next move's read;
        it is materialised here when the particles are asked for."""
        if self._pending:
            new = torch.empty(self._hi - self._lo, self.D, dtype=self.dtype, device=self.device)
            with torch.cuda.device(self.device):
                L.check(L.lib().bk_smc_shard_gather(C.byref(self._sh()), self.D, self._dt, new.data_ptr(),
                                                    stream_ptr(self.device)))
            self._src_local, self._pending = new, False
            self._check()
        return self._src_local

    @thetas.setter
    def thetas(self, value) -> None:
        self._src_local, self._pending = to_dev(value, self.dtype, self.device).clone(), False

    def log_prior(self, theta):
        return self._model.log_prior(theta)

    def log_likelihood(self, theta):
        return self._model.log_likelihood(theta)

    def __iter__(self) -> Iterator[torch.Tensor]:
        self.run()
        return iter(self.thetas)

    def run(self) -> None:
        """All N temperatures (smc.py:39-41), enqueued by ONE library call: three launches per temperature back to
        back, no Python between the steps."""
        self.run_steps(1, self.N)
        self._check()

    def run_steps(self, n_from: int, n_to: int) -> None:
        """Temperatures n_from..n_to in one library call (device Philox; injected streams go through transition())."""
        lib = L.lib()
        n_from, n_to = int(n_from), int(n_to)
        if n_to < n_from:
            return
        Ml = self._hi - self._lo
        k0 = len(self._steps_taken)
        if k0 + (n_to - n_from + 1) > self._stats.shape[0]:
            self._stats = torch.cat([self._stats, torch.zeros(n_to - n_from + 1, 4, dtype=torch.float64, device=self.device)])
        self._epoch += 1                       # epoch of step n_from
        self._acc = torch.empty(Ml, dtype=torch.int32, device=self.device)
        rng = make_rng(self._seed, n_from, self._lo, None, None, 1)
        kn = self.kernel.desc()
        src = None if self._pending else self._src_local.data_ptr()
        thr = float(self.ess_threshold) * self.M if self.ess_threshold is not None else 0.0
        with torch.cuda.device(self.device):
            L.check(lib.bk_smc_shard_run(self._model.handle, C.byref(self._sh()), src, n_from, n_to, self.N, C.byref(kn),
                                         C.byref(rng), self._mode, thr, self._stats[k0].data_ptr(), self._acc.data_ptr(),
                                         self._ws.data_ptr(), self._ws.numel(), stream_ptr(self.device)))
        self._epoch += n_to - n_from           # epoch of step n_to
        self._steps_taken.extend(range(n_from, n_to + 1))
        self._pending = True
        self.last_accept = self._acc

    def time(self, n: int) -> float:
        return n / self.N

    @property
    def weight_ess(self):
        """Importance-weight ESS (sum w)^2 / sum w^2 (over ALL ranks) per temperature taken so far.
        Diagnostic only unless ``ess_threshold`` is set: the reference resamples unconditionally (smc.py:60)."""
        if not self._steps_taken:
            return []
        s = self._stats[: len(self._steps_taken)].cpu()
        return [float(a * a / b) if b > 0 else float("nan") for _, a, b, _ in s.tolist()]

    @property
    def log_weights(self) -> torch.Tensor:
        """Unnormalised log-weights of the current particles (zeros right after a resampling)."""
        if self.ess_threshold is None or self._epoch == 0:
            return torch.zeros(self._hi - self._lo, dtype=self.dtype, device=self.device)
        return self._logw

    @property
    def resampled(self):
        """Per temperature taken so far: did the step resample?"""
        if not self._steps_taken:
            return []
        return [bool(v) for v in self._stats[: len(self._steps_taken), 3].cpu().tolist()]

    @property
    def last_indices(self) -> Optional[torch.Tensor]:
        """Resample indices (global particle ids) of this rank's slots after the last step.  With more than
        one rank they are final once every rank finished the step (``thetas`` / ``run()`` wait for that)."""
        return self._idx if self._epoch else None

    def transition(self, n: int, normals=None, acc_uniforms=None, res_uniforms=None) -> None:
        """One temperature step (smc.py:46-60).  The optional arrays inject the
        reference's recorded legacy-RNG streams (parity mode): proposal normals
        [M_local, D], accept uniforms [M_local], resampling uniforms [M_local] (systematic: [1]).
        With ``proposal_kernel``: normals [M_local, normals] and acc_uniforms [M_local, 1 + uniforms] (column 0 the
        accept uniform, columns 1.. the proposal's u; [M_local] when it draws no uniforms)."""
        self._move(n, normals, acc_uniforms)
        self._resample(n, res_uniforms, 0)

    # the two halves of a step; a FakeWorld test drives every rank through _move, then _resample(.., 1),
    # then _resample(.., 2) so that each kernel finds its messages already posted
    def _move(self, n: int, normals=None, acc_uniforms=None) -> None:
        lib = L.lib()
        Ml = self._hi - self._lo
        self._epoch += 1
        self._acc = torch.empty(Ml, dtype=torch.int32, device=self.device)
        nz, nu = self.kernel.stream_widths(self.D)
        if normals is not None and isinstance(self.kernel, ProposalKernel):
            normals = to_dev(normals, self.dtype, self.device)
            acc_uniforms = to_dev(acc_uniforms, self.dtype, self.device)
            if normals.numel() != Ml * nz or acc_uniforms.numel() != Ml * nu:
                raise ValueError(f"injected streams of the proposal move: normals [{Ml}, {nz}] and acc_uniforms "
                                 f"[{Ml}, {nu}] (got {tuple(normals.shape)} and {tuple(acc_uniforms.shape)})")
            normals, acc_uniforms = normals.reshape(Ml, nz), acc_uniforms.reshape(Ml, nu)
        elif normals is not None:
            normals = to_dev(normals, self.dtype, self.device).reshape(Ml, self.D)
            acc_uniforms = to_dev(acc_uniforms, self.dtype, self.device).reshape(Ml)
        self._inj = (normals, acc_uniforms)     # keep the injected streams alive until the kernel ran
        rng = make_rng(self._seed, n, self._lo, normals, acc_uniforms, nu)
        kn = self.kernel.desc()
        src = None if self._pending else self._src_local.data_ptr()
        accumulate = 1 if (self.ess_threshold is not None and self._epoch > 1) else 0
        with torch.cuda.device(self.device):
            L.check(lib.bk_smc_shard_move(self._model.handle, C.byref(self._sh()), src, n, self.N, C.byref(kn),
                                          C.byref(rng), accumulate, self._acc.data_ptr(), self._ws.data_ptr(),
                                          self._ws.numel(), stream_ptr(self.device)))
        self.last_accept = self._acc

    def _resample(self, n: int, res_uniforms=None, phase: int = 0) -> None:
        lib = L.lib()
        ru = None
        if res_uniforms is not None:
            ru = to_dev(res_uniforms, self.dtype, self.device).reshape(-1)
            if self._mode == L.RESAMPLE_MULTINOMIAL and ru.numel() == self.M and self._world > 1:
                ru = ru[self._lo:self._hi].contiguous()
        self._ru = ru
        rrng = make_rng(self._seed, n, 0)
        thr = float(self.ess_threshold) * self.M if self.ess_threshold is not None else 0.0
        k = len(self._steps_taken)
        with torch.cuda.device(self.device):
            L.check(lib.bk_smc_shard_resample(C.byref(self._sh()), self._dt, self._mode,
                                              None if ru is None else ru.data_ptr(), C.byref(rrng), thr, phase,
                                              self._stats[min(k, self.N)].data_ptr(), self._ws.data_ptr(),
                                              self._ws.numel(), stream_ptr(self.device)))
        if phase in (0, 2):
            self._steps_taken.append(n)
            self._pending = True    # thetas[idxs]: folded into the next move (or .thetas)

    def wire_bytes_per_step(self) -> dict:
        """Bytes this rank put on / took off NVLink in the LAST temperature step, by kind (synchronises): the three
        messages to each peer, the index stores into slots other ranks own, and the particle rows (+ their
        (ll, prior) pairs) read from peers -- counted from the step's resample indices.  Systematic resampling
        keeps most parents local (slot k's parent is particle ~k); multinomial parents are uniform over the ranks."""
        g, nl = self._world, self._hi - self._lo
        es = 4 if self.dtype == torch.float32 else 8
        out = {"messages": (16 + 32 + 8) * (g - 1), "indices": 0, "particle_rows": 0}
        if g == 1 or not self._epoch:
            return out
        if isinstance(self._group, P_.FakeRank):
            torch.cuda.synchronize(self.device)
        else:
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self._group)
        idx = self._idx
        remote_parents = int(((idx < self._lo) | (idx >= self._hi)).sum().item())
        out["particle_rows"] = remote_parents * (self.D + 2) * es
        # offspring this rank resolved for slots owned elsewhere == by symmetry of the protocol the remote parents of the
        # OTHER ranks; all-reduce the count for the exact figure, or report the local mirror (parents read remotely)
        out["indices"] = remote_parents * 8
        return out
