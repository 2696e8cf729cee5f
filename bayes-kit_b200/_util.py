"""Tensor plumbing shared by the host-side classes (torch = device memory,
streams and torch.distributed; never the compute path)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L

_DT = {torch.float32: L.BK_F32, torch.float64: L.BK_F64}


def dtype_id(dt: torch.dtype) -> int:
    try:
        return _DT[dt]
    except KeyError:
        raise TypeError(f"dtype must be torch.float32 or torch.float64, not {dt}") from None


def require_cuda(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("bayes_kit_b200 runs on CUDA devices only (no CPU fallback)")
    if not torch.cuda.is_available():
        raise RuntimeError("bayes_kit_b200: no CUDA device available (there is no CPU fallback)")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def to_dev(x, dtype, device) -> torch.Tensor:
    """array-like / tensor -> contiguous device tensor of `dtype`."""
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype).contiguous()
    return torch.as_tensor(np.asarray(x, dtype=np.float64), dtype=dtype, device=device).contiguous()


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


class Workspace:
    """Grow-only byte scratch owned by the caller side of the ABI."""

    def __init__(self, device):
        self.device = device
        self.buf = None

    def get(self, nbytes: int):
        nbytes = int(nbytes)
        if nbytes == 0:
            return None, 0
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self.buf.data_ptr(), self.buf.numel()


def compile_log(call, prefix: str, device) -> str:
    """Run ``call(log, log_bytes)``, a library entry point that compiles a user program (NVRTC) and fills its log, on
    ``device``; return the decoded log.  A compile error (``BK_E_INVALID`` with a log) raises ``ValueError(prefix +
    log)``, any other failure ``L.check``'s error."""
    log = C.create_string_buffer(1 << 20)
    with torch.cuda.device(device):
        rc = call(log, len(log))
    text = log.value.decode(errors="replace")
    if rc == L.BK_E_INVALID and text:
        raise ValueError(prefix + text)
    L.check(rc)
    return text


def make_rng(seed, draw_offset, chain_offset, normals=None, uniforms=None, n_uniform=1) -> L.Rng:
    r = L.Rng()
    if normals is not None or uniforms is not None:
        if normals is None or uniforms is None:
            raise ValueError("injected streams need both normals and uniforms")
        r.mode = L.RNG_INJECTED
        r.normals, r.uniforms = normals.data_ptr(), uniforms.data_ptr()
        r.n_uniform = n_uniform
    else:
        r.mode = L.RNG_PHILOX
        r.n_uniform = n_uniform
    r.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    r.draw_offset = int(draw_offset)
    r.chain_offset = int(chain_offset)
    return r


def resolve_seed(seed) -> int:
    """Reference: np.random.default_rng(seed) (hmc.py:23).  None -> fresh entropy."""
    if seed is None:
        return int(np.random.SeedSequence().generate_state(2, dtype=np.uint32).view(np.uint64)[0])
    if isinstance(seed, (int, np.integer)):
        return int(seed)
    if isinstance(seed, np.random.Generator):
        return int(seed.integers(0, 2**63 - 1))
    if isinstance(seed, np.random.BitGenerator):
        return int(np.random.Generator(seed).integers(0, 2**63 - 1))
    raise TypeError(f"seed must be None, an int, a BitGenerator or a Generator, not {type(seed)}")
