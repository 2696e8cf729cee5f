"""Shared host logic of the lockstep MCMC samplers (one object == C chains)."""
from __future__ import annotations

from typing import Iterator, Optional, Tuple

import torch

from . import _lib as L
from ._util import Workspace, make_rng, ptr, resolve_seed, stream_ptr, to_dev
from .models import require_plugin

DrawAndLogP = Tuple[torch.Tensor, torch.Tensor]


def _is_empty_init(init) -> bool:
    # reference: `init is not None and init.shape != (0,)` (hmc.py:24-28)
    return init is None or tuple(getattr(init, "shape", (1,))) == (0,)


class ChainSampler:
    """C independent chains advanced in lockstep on one GPU.

    ``init`` of shape [D] keeps the reference's single-chain surface
    (``sample() -> (theta[D], logp)``); shape [C, D] (or ``chains=C``) runs C
    chains and ``sample()`` returns ``(Theta[C, D], logp[C])``.  Randomness is
    device Philox keyed by (seed, global chain id, draw index) -- results do
    not depend on how chains are sharded over GPUs -- unless pre-drawn streams
    are injected (``sample_n(n, normals=..., uniforms=...)``, parity mode).
    """

    _n_uniform = 1

    def __init__(self, model, init, seed, chains: Optional[int], chain_offset: int = 0):
        self._model = require_plugin(model)
        self._dim = self._model.dims()
        self._n_normal = self._dim   # injected normals per (draw, chain)
        self.device, self.dtype = self._model.device, self._model.dtype
        self._seed = resolve_seed(seed)
        self._chain_offset = int(chain_offset)
        self._t = 0  # draws taken so far (Philox draw counter)
        if _is_empty_init(init):
            n = 1 if chains is None else int(chains)
            self._single = chains is None
            # theta0 ~ N(0, I) like rng.normal(size=dim) (hmc.py:27): device Philox keyed by the GLOBAL chain id
            th = self._philox_normal(n, 0xFFFFFFFF)
        else:
            th = to_dev(init, self.dtype, self.device)
            self._single = th.dim() == 1
            th = th.reshape(1, -1) if self._single else th
            if th.dim() != 2 or th.shape[1] != self._dim:
                raise ValueError(f"init must have shape [{self._dim}] or [C, {self._dim}], "
                                 f"got {tuple(th.shape)}")
            if chains is not None and int(chains) != th.shape[0]:
                raise ValueError("chains does not match init.shape[0]")
            th = th.clone()
        self._theta = th.contiguous()
        self._C = self._theta.shape[0]
        self._ws = Workspace(self.device)
        self._lp = torch.empty(self._C, dtype=self.dtype, device=self.device)
        self._grad = None
        self._cache_valid = L.i32(0)
        self.last_accept = None

    def _philox_normal(self, n: int, draw: int) -> torch.Tensor:
        """[n, D] standard normals for global chains chain_offset .. chain_offset + n (shard invariant)."""
        out = torch.empty(n, self._dim, dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            L.check(L.lib().bk_init_normal(out.data_ptr(), n, self._dim, L.BK_F32 if self.dtype == torch.float32 else L.BK_F64,
                                           self._seed & 0xFFFFFFFFFFFFFFFF, self._chain_offset, draw, stream_ptr(self.device)))
        return out

    # ---- reference surface ---------------------------------------------------------
    def __iter__(self) -> Iterator[DrawAndLogP]:
        return self

    def __next__(self) -> DrawAndLogP:
        return self.sample()

    def sample(self) -> DrawAndLogP:
        draws, logp = self.sample_n(1)
        return draws[0], logp[0]

    # ---- batched extension -----------------------------------------------------------
    @property
    def chains(self) -> int:
        return self._C

    @property
    def theta(self) -> torch.Tensor:
        return self._theta[0] if self._single else self._theta

    def _fuses_extras(self) -> bool:
        """True when this sampler's engine folds streaming moments / writes series-major draws inside its own
        kernel: the fp32 register-resident samplers of the iso / diagonal Gaussian plugins (bk.h: bk_draw_out)."""
        from .models import DiagGauss, IsoGauss
        import os
        return (self.dtype == torch.float32 and isinstance(self._model, (IsoGauss, DiagGauss)) and self._dim <= 512
                and os.environ.get("BK_FORCE_GENERIC", "0") != "1" and type(self).__name__ != "DrGhmcDiag")

    def sample_n(self, n: int, normals=None, uniforms=None, keep_draws: bool = True, moments: bool = False,
                 layout: str = "draws"):
        """Advance every chain n draws in one call.  Returns (draws [n, C, D],
        logp [n, C]) ([n, D], [n] for a single chain); with keep_draws=False only
        the final state is kept (warm-up) and draws is None.  ``moments=True``
        folds the batch into running per-chain, per-dimension mean / variance
        (``running_moments()``, ``running_rhat()``) -- convergence monitoring
        without storing or re-reading the chains: the fused fp32 samplers accumulate in
        registers inside the sampling kernel (no second pass), the GEMM engines fold the
        draws they wrote.  ``layout="series"`` (fused fp32 samplers): draws come back as
        [C, D, n] -- every (chain, dim) series contiguous over the draws, the layout
        ``ess`` / ``iat`` / ``autocorr`` stream without a transposition (SURVEY 8(f)-2)."""
        n = int(n)
        C_, D = self._C, self._dim
        if layout not in ("draws", "series"):
            raise ValueError("layout must be 'draws' ([n, C, D]) or 'series' ([C, D, n])")
        fused = self._fuses_extras()
        if layout == "series" and not fused:
            raise NotImplementedError("layout='series' is written by the fused fp32 samplers of the iso / diagonal "
                                      "Gaussian plugins; other engines return [n, C, D] (diagnostics read it in place)")
        need_buf = keep_draws or (moments and not fused)
        if moments and not keep_draws and not fused and n > 16:      # bound the transient draw buffer
            out_l = []
            for k in range(0, n, 16):
                out_l.append(self.sample_n(min(16, n - k), keep_draws=False, moments=True)[1])
            return None, torch.cat(out_l)
        shape = (C_, D, n) if layout == "series" else (n, C_, D)
        draws = torch.empty(*shape, dtype=self.dtype, device=self.device) if need_buf else None
        logp = torch.empty(n, C_, dtype=self.dtype, device=self.device)
        acc = torch.empty(n, C_, dtype=torch.int32, device=self.device)
        if normals is not None:
            normals = to_dev(normals, self.dtype, self.device).reshape(n, C_, self._n_normal)
            uniforms = to_dev(uniforms, self.dtype, self.device).reshape(n, C_, self._n_uniform)
        rng = make_rng(self._seed, self._t, self._chain_offset, normals, uniforms, self._n_uniform)
        out = L.DrawOut(ptr(draws), logp.data_ptr(), acc.data_ptr())
        out.layout = L.DRAWS_CDN if layout == "series" else L.DRAWS_NCD
        if moments and n > 0:
            if getattr(self, "_mom", None) is None:
                self._mom = [torch.empty(C_, D, dtype=torch.float64, device=self.device),
                             torch.empty(C_, D, dtype=torch.float64, device=self.device), 0]
            if type(self).__name__ != "DrGhmcDiag":       # folded by the library (in-kernel where the engine fuses it)
                out.mom_mean, out.mom_m2, out.mom_n0 = self._mom[0].data_ptr(), self._mom[1].data_ptr(), self._mom[2]
        with torch.cuda.device(self.device):
            self._launch(n, rng, out)
            if moments and n > 0 and type(self).__name__ == "DrGhmcDiag":
                L.check(L.lib().bk_moments_accumulate(
                    draws.data_ptr(), L.BK_F32 if self.dtype == torch.float32 else L.BK_F64, n, C_ * D,
                    self._mom[2], self._mom[0].data_ptr(), self._mom[1].data_ptr(), stream_ptr(self.device)))
        self._t += n
        self.last_accept = acc[:, 0] if self._single else acc
        if moments and n > 0:
            self._mom[2] += n
            if not keep_draws:
                draws = None
        if self._single:
            if draws is not None:
                draws = draws[0] if layout == "series" else draws[:, 0]
            return draws, logp[:, 0]
        return draws, logp

    def running_moments(self):
        """(mean [C, D], var [C, D] with ddof=1, n) over every draw taken with
        ``moments=True`` so far (fp64)."""
        if getattr(self, "_mom", None) is None or self._mom[2] < 2:
            raise ValueError("running moments need at least 2 draws taken with moments=True")
        return self._mom[0], self._mom[1] / (self._mom[2] - 1), self._mom[2]

    def running_rhat(self) -> torch.Tensor:
        """R-hat per dimension (rhat.py:111-171) from the running moments of this
        sampler's chains: no pass over stored draws."""
        from .rhat import _rhat_from
        mean, var, n = self.running_moments()
        return _rhat_from(mean, var, None, n)

    def reset_moments(self) -> None:
        self._mom = None

    def sample_host(self, theta_host=None, out=None, chunk_chains=None):
        """One draw of every chain with HOST buffers, pipelined over chain chunks.

        The reference's ``sample()`` hands back host arrays (hmc.py:63); this is
        that call for C lockstep chains without serialising on PCIe: chains are
        cut into chunks and chunk k's device->host copy of its draw, chunk
        k+1's kernels and chunk k+2's host->device copy of its state run
        concurrently on three streams.  Chunking cannot change the result --
        Philox is keyed by the global chain id.

        theta_host  [C, D] host tensor (pinned for overlap): the chain state is
                    loaded from it first (and the cached log density / gradient
                    recomputed); None keeps the device-resident state.
        out         (draw_host [C, D], logp_host [C]) pinned tensors to fill;
                    allocated (pinned) when None.
        chunk_chains  chains per chunk (default: 37 chain-tiles of 256 at D ~ 1000) or an explicit
                    list of chunk sizes summing to C.  Setting ``self._trace = []`` beforehand
                    collects (stream, chunk, start, end) CUDA events of the three streams.
        Returns (draw_host, logp_host), complete on return; ``theta`` holds the
        same draw on device and ``last_accept`` the accept flags.
        """
        if self._single:
            raise ValueError("sample_host is the batched surface: construct with init [C, D] or chains=C")
        C_, D = self._C, self._dim
        if out is None:
            out = (torch.empty(C_, D, dtype=self.dtype).pin_memory(),
                   torch.empty(C_, dtype=self.dtype).pin_memory())
        draw_h, logp_h = out
        for name, t, shape in (("theta_host", theta_host, (C_, D)), ("out[0]", draw_h, (C_, D)),
                               ("out[1]", logp_h, (C_,))):
            if t is not None and (tuple(t.shape) != shape or t.dtype != self.dtype or t.is_cuda
                                  or not t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous host {self.dtype} tensor of shape {shape}")
        if isinstance(chunk_chains, (list, tuple)):     # explicit chunk sizes
            sizes = [int(c) for c in chunk_chains]
            if any(c <= 0 for c in sizes) or sum(sizes) != C_:
                raise ValueError(f"chunk sizes must be positive and sum to {C_}")
        else:
            if chunk_chains is None:
                # 37 chain-tiles of 256 (two full waves of the 148-CTA gradient GEMM) at D ~ 1000
                chunk_chains = max(256, int(round(9472 * 1000 / max(D, 1) / 256)) * 256)
            chunk_chains = max(1, min(int(chunk_chains), C_))
            sizes = []
            c = sum(sizes)
            while c < C_:
                sizes.append(min(chunk_chains, C_ - c))
                c += sizes[-1]
        if getattr(self, "_hs", None) is None:
            self._hs = tuple(torch.cuda.Stream(self.device) for _ in range(3))
            self._h_draw = torch.empty(C_, D, dtype=self.dtype, device=self.device)
            self._h_logp = torch.empty(C_, dtype=self.dtype, device=self.device)
            self._h_acc = torch.empty(C_, dtype=torch.int32, device=self.device)
        s_in, s_run, s_out = self._hs
        cur = torch.cuda.current_stream(self.device)
        for s in self._hs:
            s.wait_stream(cur)
        # state loaded from the host (or never evaluated): the (logp, grad) cache is stale
        stale = theta_host is not None or not self._cache_valid.value
        # optional timeline (scripts/e2e_sweep.py): self._trace = [] collects (stream, chunk, start, end) events
        trace = getattr(self, "_trace", None)

        def mark(stream):
            if trace is None:
                return None
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            return e
        c0 = 0
        for k, cn in enumerate(sizes):
            valid = L.i32(0 if stale else 1)
            if theta_host is not None:
                with torch.cuda.stream(s_in):
                    t0 = mark(s_in)
                    self._theta[c0:c0 + cn].copy_(theta_host[c0:c0 + cn], non_blocking=True)
                    if trace is not None:
                        trace.append(("h2d", k, t0, mark(s_in)))
                s_run.wait_stream(s_in)
            with torch.cuda.stream(s_run):
                rng = make_rng(self._seed, self._t, self._chain_offset + c0, None, None, self._n_uniform)
                o = L.DrawOut(self._h_draw[c0:].data_ptr(), self._h_logp[c0:].data_ptr(),
                              self._h_acc[c0:].data_ptr())
                t0 = mark(s_run)
                self._launch(1, rng, o, c0, cn, valid)
                done = torch.cuda.Event(enable_timing=trace is not None)
                done.record(s_run)
                if trace is not None:
                    trace.append(("run", k, t0, done))
            s_out.wait_event(done)
            with torch.cuda.stream(s_out):
                t0 = mark(s_out)
                draw_h[c0:c0 + cn].copy_(self._h_draw[c0:c0 + cn], non_blocking=True)
                logp_h[c0:c0 + cn].copy_(self._h_logp[c0:c0 + cn], non_blocking=True)
                if trace is not None:
                    trace.append(("d2h", k, t0, mark(s_out)))
            c0 += cn
        self._t += 1
        self.last_accept = self._h_acc
        self._cache_valid.value = 1              # every chunk refreshed its slice of the cache
        cur.wait_stream(s_run)
        s_out.synchronize()
        return draw_h, logp_h

    def sample_host_n(self, n: int, theta_host=None, out=None, chunk_chains=None):
        """``n`` draws of every chain with HOST buffers -- what a caller of the reference ends up with after
        ``[sampler.sample() for _ in range(n)]`` (host arrays, hmc.py:63): the chain state goes in ONCE
        (``theta_host`` [C, D], optional), all n draws and log densities come back
        (``out = (draws_host [n, C, D], logp_host [n, C])``, pinned; allocated when None).  The pipeline runs over
        DRAWS: draw t's device->host copy overlaps draw t+1's kernels (all chains at once, a ring of three device
        staging buffers); only the first draw is cut into chain chunks so that the host->device copy of the state
        overlaps its kernels.  Neither can change the result (Philox is keyed by global chain id and draw index).  Returns (draws_host, logp_host), complete on
        return; ``last_accept`` [n, C] stays on the device."""
        if self._single:
            raise ValueError("sample_host_n is the batched surface: construct with init [C, D] or chains=C")
        n = int(n)
        C_, D = self._C, self._dim
        if out is None:
            out = (torch.empty(n, C_, D, dtype=self.dtype).pin_memory(), torch.empty(n, C_, dtype=self.dtype).pin_memory())
        draws_h, logp_h = out
        for name, t, shape in (("theta_host", theta_host, (C_, D)), ("out[0]", draws_h, (n, C_, D)),
                               ("out[1]", logp_h, (n, C_))):
            if t is not None and (tuple(t.shape) != shape or t.dtype != self.dtype or t.is_cuda
                                  or not t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous host {self.dtype} tensor of shape {shape}")
        if isinstance(chunk_chains, (list, tuple)):
            sizes = [int(c) for c in chunk_chains]
            if any(c <= 0 for c in sizes) or sum(sizes) != C_:
                raise ValueError(f"chunk sizes must be positive and sum to {C_}")
        else:
            if chunk_chains is None:
                chunk_chains = max(256, int(round(9472 * 1000 / max(D, 1) / 256)) * 256)
            chunk_chains = max(1, min(int(chunk_chains), C_))
            sizes = [min(chunk_chains, C_ - c) for c in range(0, C_, chunk_chains)]
        # Pipeline over DRAWS: the device -> host copy of draw t (C * D * 4 bytes) runs while draw t + 1 is computed for
        # ALL chains at full kernel efficiency; only the first draw is chunked over chains, so that the host -> device
        # copy of the state overlaps its kernels.  The D2H stream is the critical path (a draw leaves in ~4.8 ms over
        # PCIe 5 x16, its kernels take ~3 ms at c2) and it starts after ~one chunk of the first draw.
        ring = getattr(self, "_hn_ring", None)
        if ring is None:
            ring = [(torch.empty(C_, D, dtype=self.dtype, device=self.device),
                     torch.empty(C_, dtype=self.dtype, device=self.device)) for _ in range(3)]
            self._hn_ring = ring
        if getattr(self, "_hs", None) is None:
            self._hs = tuple(torch.cuda.Stream(self.device) for _ in range(3))
        s_in, s_run, s_out = self._hs
        cur = torch.cuda.current_stream(self.device)
        for st in self._hs:
            st.wait_stream(cur)
        stale = theta_host is not None or not self._cache_valid.value
        acc_all = torch.empty(n, C_, dtype=torch.int32, device=self.device)
        freed = [None, None, None]      # event: the ring slot's previous contents have left for the host
        for t in range(n):
            slot = t % 3
            sd, sl = ring[slot]
            if freed[slot] is not None:
                s_run.wait_event(freed[slot])
            if t == 0:
                c0 = 0
                for k, cn in enumerate(sizes):
                    valid = L.i32(0 if stale else 1)
                    if theta_host is not None:
                        with torch.cuda.stream(s_in):
                            self._theta[c0:c0 + cn].copy_(theta_host[c0:c0 + cn], non_blocking=True)
                        s_run.wait_stream(s_in)
                    with torch.cuda.stream(s_run):
                        rng = make_rng(self._seed, self._t, self._chain_offset + c0, None, None, self._n_uniform)
                        o = L.DrawOut(sd[c0:].data_ptr(), sl[c0:].data_ptr(), acc_all[0, c0:].data_ptr())
                        self._launch(1, rng, o, c0, cn, valid)
                        done = torch.cuda.Event()
                        done.record(s_run)
                    s_out.wait_event(done)
                    with torch.cuda.stream(s_out):
                        draws_h[0, c0:c0 + cn].copy_(sd[c0:c0 + cn], non_blocking=True)
                        logp_h[0, c0:c0 + cn].copy_(sl[c0:c0 + cn], non_blocking=True)
                    c0 += cn
                self._cache_valid.value = 1
            else:
                with torch.cuda.stream(s_run):
                    rng = make_rng(self._seed, self._t + t, self._chain_offset, None, None, self._n_uniform)
                    o = L.DrawOut(sd.data_ptr(), sl.data_ptr(), acc_all[t].data_ptr())
                    self._launch(1, rng, o, 0, C_, L.i32(1))
                    done = torch.cuda.Event()
                    done.record(s_run)
                s_out.wait_event(done)
                with torch.cuda.stream(s_out):
                    draws_h[t].copy_(sd, non_blocking=True)
                    logp_h[t].copy_(sl, non_blocking=True)
            with torch.cuda.stream(s_out):
                ev = torch.cuda.Event()
                ev.record(s_out)
                freed[slot] = ev
        self._t += n
        self.last_accept = acc_all
        self._cache_valid.value = 1
        cur.wait_stream(s_run)
        s_out.synchronize()
        return draws_h, logp_h

    def _launch(self, n, rng, out, c0=0, cn=None, cache_valid=None):  # pragma: no cover - overridden
        raise NotImplementedError

    def _need_grad_cache(self):
        if self._grad is None:
            self._grad = torch.empty_like(self._theta)
