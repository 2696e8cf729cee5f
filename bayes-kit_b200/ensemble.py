"""Stretcher -- affine-invariant ensemble sampler (reference: bayes_kit/ensemble.py).

Upstream the class body is a docstring only: the Goodman & Weare stretch-move
implementation is commented out (ensemble.py:16-66).  This is that algorithm, with
the constructor the comments sketch, running on device: the walkers of one half
move in parallel against the complementary half (three launches per half-step,
the density through the model plugin -- tensor cores where it has them; one
fused launch, compiled from the model's source, for a ``CudaModel`` /
``CudaPriorLikModel`` with ``dims <= 32``).  With
torch.distributed initialised each rank owns a slice of both halves and the
complementary half is all-gathered before each half-step (the one collective).
Parity is pinned by oracle/samplers.py::stretch only (no executable reference).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from . import dist as D_
from . import peer as P_
from ._util import Workspace, compile_log, make_rng, resolve_seed, stream_ptr, to_dev
from .models import CudaModel, require_plugin


class Stretcher:
    """``Stretcher(model, a=None, walkers=None, init=None)`` (ensemble.py:16-40).

    * ``a``: stretch bound >= 1 (default 2, Goodman & Weare's choice).
    * ``walkers``: strictly positive even integer, default ``2 * dims``.
    * ``init``: ``[walkers, dims]``; default ``N(0, I)`` draws (ensemble.py:38).
    ``sample()`` performs one sweep (first half against the second, then the second
    against the updated first, ensemble.py:55-63) and returns the walkers
    ``[walkers, dims]`` (this rank's walkers under torch.distributed).
    On a ``CudaModel`` / ``CudaPriorLikModel`` with ``dims <= 32`` each half-step
    is one fused kernel compiled from the model's source at construction
    (``compile_log``: ptxas's report, ``""`` on every other engine; a compile
    error raises ``ValueError`` with NVRTC's log).
    """

    def __init__(self, model, a: Optional[float] = None, walkers: Optional[int] = None, init=None, *,
                 seed=None, group=None):
        self._model = require_plugin(model)
        self._dim = self._model.dims()
        self.device, self.dtype = self._model.device, self._model.dtype
        if a is not None and a < 1:
            raise ValueError(f"stretch bound must be greater than or equal to 1; found {a=}")
        self._a = 2.0 if a is None else float(a)
        if walkers is not None and (not isinstance(walkers, (int, np.integer)) or walkers <= 0 or walkers % 2 != 0):
            raise ValueError(f"walkers must be strictly positive, even integer; found {walkers=}")
        self._walkers = int(walkers) if walkers is not None else 2 * self._dim
        self._halfwalkers = self._walkers // 2
        self._drawshape = (self._walkers, self._dim)
        if init is not None and tuple(init.shape) != self._drawshape:
            raise ValueError(f"init must be shape of draw {self._drawshape}; found init.shape={tuple(init.shape)}")
        self._seed = resolve_seed(seed)
        self._group = group
        self._rank, self._world = P_.rank_world(group)
        if init is not None:
            th = to_dev(init, self.dtype, self.device).clone()
        else:
            g = torch.Generator(device=self.device)
            g.manual_seed(self._seed % (2 ** 63))
            th = torch.randn(*self._drawshape, generator=g, device=self.device, dtype=self.dtype)
        # this rank's slice of each half (global walker ids lo..hi within the half)
        h = self._halfwalkers
        self._lo, self._hi = D_.shard_range(h, self._rank, self._world)
        self._halves = [th[:h][self._lo:self._hi].contiguous(), th[h:][self._lo:self._hi].contiguous()]
        nl = self._hi - self._lo
        self._lp = [torch.empty(nl, dtype=self.dtype, device=self.device) for _ in range(2)]
        self._valid = [L.i32(0), L.i32(0)]
        self._ws = Workspace(self.device)
        self._t = 0
        self.last_accept = None
        self.compile_log = ""
        if isinstance(self._model, CudaModel):
            # compile the fused kernel now, not in the first sample(); its log, or "" (three-launch engine)
            self.compile_log = compile_log(
                lambda log, n: L.lib().bk_stretch_cuda_prepare(self._model.handle, log, n),
                "Stretcher: NVRTC compilation of the model's stretch kernel failed:\n", self.device)
        if isinstance(group, P_.FakeRank):      # single-GPU fake world: the other ranks' halves live on this device
            group.fake._regions.setdefault("stretch", [None] * self._world)[self._rank] = self._halves

    def __iter__(self):
        return self

    def __next__(self):
        return self.sample()

    @property
    def thetas(self) -> torch.Tensor:
        """This rank's walkers [first-half slice; second-half slice]."""
        return torch.cat(self._halves)

    def sample(self, uniforms=None) -> torch.Tensor:
        """One sweep.  ``uniforms`` [walkers, 3] injects (partner, stretch, accept)
        uniforms per walker (parity mode; this rank's rows under torch.distributed)."""
        for half in (0, 1):
            self._half_step(half, uniforms)
        return self.thetas

    def _half_step(self, half: int, uniforms=None) -> None:
        """Move this rank's walkers of one half against the complementary half (ensemble.py:55-63).  A
        FakeWorld test calls this for every rank before moving on to the other half."""
        lib = L.lib()
        nl = self._hi - self._lo
        h = self._halfwalkers
        if half == 0:
            self._acc = torch.empty(2, nl, dtype=torch.int32, device=self.device)
        if uniforms is not None:
            uniforms = to_dev(uniforms, self.dtype, self.device).reshape(2, nl, 3)
        with torch.cuda.device(self.device):
            wp, wn = self._ws.get(lib.bk_stretch_workspace_bytes(self._model.handle, nl))
            other = self._complement(half)                                        # complementary walkers [h, D]
            rng = make_rng(self._seed, 2 * self._t + half, half * h + self._lo, None, None, 3)
            if uniforms is not None:
                rng.mode, rng.uniforms = L.RNG_INJECTED, uniforms[half].data_ptr()
            L.check(lib.bk_stretch_move(
                self._model.handle, self._halves[half].data_ptr(), self._lp[half].data_ptr(),
                C.byref(self._valid[half]), other.data_ptr(), nl, other.shape[0], self._a, C.byref(rng),
                self._acc[half].data_ptr(), wp, wn, stream_ptr(self.device)))
        if half == 1:
            self._t += 1
            self.last_accept = self._acc.reshape(-1)

    def _complement(self, half: int) -> torch.Tensor:
        """All walkers of the half that is NOT being moved: all-gather of every rank's slice (sizes are
        known from the shard rule -> no size exchange, no host sync).  FakeWorld: the other ranks'
        slices live on this device."""
        mine = self._halves[1 - half]
        if isinstance(self._group, P_.FakeRank):
            reg = self._group.fake._regions["stretch"]
            if any(r is None for r in reg):
                raise RuntimeError("FakeWorld: construct every rank before sampling")
            return torch.cat([r[1 - half] for r in reg])
        return D_.all_gather_cat(mine, self._group, sizes=D_.shard_sizes(self._halfwalkers, self._world))

    def sample_n(self, n: int) -> torch.Tensor:
        """n sweeps -> draws [n, walkers_local, dims]."""
        return torch.stack([self.sample().clone() for _ in range(int(n))])
