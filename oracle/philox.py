"""NumPy restatement of the device random streams (``bayes-kit_b200/csrc/device_rng.cuh``).

TEST INFRASTRUCTURE (see oracle/__init__.py).

Philox4x32-10 (Salmon et al. 2011) with counter ``(block, tag, chain, draw)``
and key ``seed`` (low word, high word), the uniform grids ``u01`` / ``u01d``,
``philox_uniform``, the accept-uniform rule of the single-uniform samplers,
the fp64 normals of ``philox_normal4<double>`` and the fp32 Box-Muller of
``box_muller4``.  Every function is vectorised over NumPy arrays of counter
words.  The fp32 Box-Muller is evaluated here in fp64 from the same fp32
inputs; the device uses ``lg2.approx`` / ``sin.approx`` / ``cos.approx``, so
it matches the device only to the error of those instructions
(``box_muller4_tolerance``).
"""
from __future__ import annotations

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
TAG_NORMAL, TAG_NORMAL_HI, TAG_UNIFORM, TAG_RESAMPLE = 0, 1, 2, 3
_MASK = np.uint64(0xFFFFFFFF)


def _u32(x):
    return np.asarray(x, dtype=np.uint64) & _MASK


def philox4x32_10(ctr, key):
    """Philox4x32-10 on counters ``ctr = (c0, c1, c2, c3)`` and key ``(k0, k1)`` (words broadcast against
    each other).  Returns the four output words as uint32 arrays."""
    c = [_u32(w) for w in ctr]
    c = np.broadcast_arrays(*c, _u32(key[0]), _u32(key[1]))
    c, k0, k1 = [w.copy() for w in c[:4]], c[4].copy(), c[5].copy()
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]          # < 2^64: exact in uint64
        p1 = np.uint64(M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(W0)) & _MASK
        k1 = (k1 + np.uint64(W1)) & _MASK
    return [w.astype(np.uint32) for w in c]


def gen(seed, block, tag, chain, draw):
    """``Philox::gen``: counter (block, tag, chain, draw), key = (seed & 0xffffffff, seed >> 32)."""
    seed = np.asarray(seed, dtype=np.uint64)
    return philox4x32_10((block, tag, chain, draw), (seed & _MASK, seed >> np.uint64(32)))


def u01(x):
    """fp32 uniform of one word: midpoint of the 2^-23 grid, strictly inside (0, 1)."""
    x = np.asarray(x, dtype=np.uint32)
    return (((x >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(1.1920928955078125e-7)).astype(np.float32)


def u01d(hi, lo):
    """fp64 uniform of two words: midpoint of the 2^-52 grid, strictly inside (0, 1)."""
    hi, lo = np.asarray(hi, dtype=np.uint32), np.asarray(lo, dtype=np.uint32)
    return ((hi >> np.uint32(6)).astype(np.float64) * 67108864.0 + (lo >> np.uint32(6)).astype(np.float64) + 0.5) \
        * 2.220446049250313e-16


def philox_uniform(seed, k, chain, draw, dtype=np.float32, tag=TAG_UNIFORM):
    """k-th uniform of (chain, draw): fp32 = word k & 3 of block k >> 2, fp64 = word pair k & 1 of block k >> 1."""
    k = np.asarray(k, dtype=np.uint64)
    if np.dtype(dtype) == np.float32:
        r = gen(seed, k >> np.uint64(2), tag, chain, draw)
        return np.choose((k & np.uint64(3)).astype(np.int64), [u01(w) for w in r])
    r = gen(seed, k >> np.uint64(1), tag, chain, draw)
    return np.where((k & np.uint64(1)) == 1, u01d(r[2], r[3]), u01d(r[0], r[1]))


def accept_block(D):
    """First element block of the normal stream that no element of a D-dim proposal uses."""
    return (int(D) + 3) >> 2


def accept_uniform(seed, chain, draw, D, dtype=np.float32):
    """Accept uniform of HMC / MALA / RW-Metropolis in Philox mode: word 0 (fp32) or words 0, 1 (fp64) of block
    accept_block(D) of the TAG_NORMAL stream."""
    r = gen(seed, accept_block(D), TAG_NORMAL, chain, draw)
    return u01(r[0]) if np.dtype(dtype) == np.float32 else u01d(r[0], r[1])


def _sincospi(x):
    # sin / cos of pi x for x in (0, 2), reduced to |x| <= 1/4 so that no precision is lost to the argument
    x = np.asarray(x, dtype=np.float64)
    n = np.rint(2.0 * x)
    r = (x - 0.5 * n) * np.pi
    s, c = np.sin(r), np.cos(r)
    q = n.astype(np.int64) & 3
    sin = np.choose(q, [s, c, -s, -c])
    cos = np.choose(q, [c, -s, -c, s])
    return sin, cos


def normal4_f64(seed, block, chain, draw):
    """``philox_normal4<double>``: the 4 normals of element block `block`, shape [4, ...]."""
    a = gen(seed, block, TAG_NORMAL, chain, draw)
    b = gen(seed, block, TAG_NORMAL_HI, chain, draw)
    r0 = np.sqrt(-2.0 * np.log(u01d(a[0], a[1])))
    r1 = np.sqrt(-2.0 * np.log(u01d(b[0], b[1])))
    s0, c0 = _sincospi(2.0 * u01d(a[2], a[3]))
    s1, c1 = _sincospi(2.0 * u01d(b[2], b[3]))
    return np.stack([r0 * c0, r0 * s0, r1 * c1, r1 * s1])


def _bm_radius(w):
    # u = fmaf(float(w), 2^-32, 2^-33): the product and sum are exact in fp64, one rounding to fp32
    wf = np.asarray(w, dtype=np.uint32).astype(np.float32).astype(np.float64)
    u = (wf * 2.0 ** -32 + 2.0 ** -33).astype(np.float32).astype(np.float64)
    return np.sqrt(-2.0 * np.log(u))


def _bm_angle(w):
    # the word read as a signed integer, rounded to fp32, times 2 pi / 2^32 (rounded to fp32)
    wf = np.asarray(w, dtype=np.uint32).view(np.int32).astype(np.float32)
    return (wf * np.float32(1.4629180792671596e-9)).astype(np.float64)


def normal4_f32(seed, block, chain, draw):
    """``box_muller4`` of block `block`, evaluated in fp64 from the device's fp32 inputs: shape [4, ...]."""
    r = gen(seed, block, TAG_NORMAL, chain, draw)
    r0, r1 = _bm_radius(r[0]), _bm_radius(r[2])
    a0, a1 = _bm_angle(r[1]), _bm_angle(r[3])
    return np.stack([r0 * np.cos(a0), r0 * np.sin(a0), r1 * np.cos(a1), r1 * np.sin(a1)])


def box_muller4_tolerance(z):
    """Absolute bound on |device - normal4_f32| for a normal of magnitude |z|.  lg2.approx has absolute error
    about 2^-22 near u = 1, and r = sqrt(-2 ln u) turns an error e of ln u into e / r in r: 2^-22 / r.  sin / cos.approx
    add about 2^-20.9 absolute times r; the fp32 roundings of the radius, the angle and the product about 2^-23 r."""
    r = np.abs(np.asarray(z, dtype=np.float64))
    return 2.0 ** -21 / np.maximum(r, 1e-3) + 2.0 ** -19 * (1.0 + r)


def init_normal(seed, chain_offset, draw, C, D, dtype=np.float64):
    """[C, D] normals of ``bk_init_normal``: element e of chain c is word e % 4 of block e // 4 for global chain
    chain_offset + c."""
    nb = accept_block(D)
    blk = np.arange(nb, dtype=np.uint64)[None, :]
    ch = (np.uint64(chain_offset) + np.arange(C, dtype=np.uint64))[:, None]
    f = normal4_f64 if np.dtype(dtype) == np.float64 else normal4_f32
    z = f(seed, blk, ch, draw)                         # [4, C, nb]
    return np.moveaxis(z, 0, -1).reshape(C, 4 * nb)[:, :D]
