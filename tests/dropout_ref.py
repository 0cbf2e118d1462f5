"""Host reference of the counter-based dropout RNG that every mask of the library follows (nnr_b200/csrc/common.cuh).

Element ``i`` of a tensor dropped with ``(seed, p)`` uses 16-bit field ``i & 3`` of
``mix64(seed * 0x9E3779B97F4A7C15 + (i >> 2))`` (all mod 2^64): it is dropped when that field is below
``uint32(float32(p) * 65536)``, and a kept element is scaled by ``float32(1) / (float32(1) - float32(p))``.  A seed with
bit 62 set is indirect: bits 0..47 hold the device address of a uint64 base, bits 48..61 a site id, and the kernels use
``mix64(base + site * 0x9E3779B97F4A7C15) >> 2``.

Everything here is integer arithmetic on the host, independent of the kernels, so a test can pin every mask bit for bit.
Arrays are numpy uint64, whose arithmetic wraps silently; scalar constants are Python ints masked to 64 bits (numpy
scalar overflow warns).
"""
import numpy as np

MASK64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15
INDIRECT = 1 << 62
_M1, _M2 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53


def mix64_int(x):
    """mix64 of common.cuh on one Python int (the scalar definition the vectorised one is checked against)"""
    x &= MASK64
    x ^= x >> 33
    x = (x * _M1) & MASK64
    x ^= x >> 33
    x = (x * _M2) & MASK64
    x ^= x >> 33
    return x


def mix64(x):
    """mix64 of common.cuh, element-wise on a numpy uint64 array"""
    x = np.asarray(x, dtype=np.uint64)
    s33 = np.uint64(33)
    x = x ^ (x >> s33)
    x = x * np.uint64(_M1)
    x = x ^ (x >> s33)
    x = x * np.uint64(_M2)
    return x ^ (x >> s33)


def resolve_indirect(base, site):
    """the seed an indirect site resolves to on the device: mix64(base + site * golden) >> 2"""
    return mix64_int((int(base) + int(site) * GOLDEN) & MASK64) >> 2


def resolve_seed(seed, base=None):
    """the seed the kernels use: a direct seed (< 2^62) as is; an indirect one through ``base`` (the uint64 it points to)"""
    seed = int(seed) & MASK64
    if seed & INDIRECT:
        assert base is not None, 'an indirect seed needs the value of its base'
        return resolve_indirect(base, (seed >> 48) & 0x3FFF)
    return seed


def threshold(p):
    """the 16-bit drop threshold: (uint32_t)(p * 65536.0f) in float32"""
    return int(np.float32(p) * np.float32(65536.0))


def inv_keep(p):
    """the scale of a kept element, 1.0f / (1.0f - p) in float32"""
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


def keep_scale(seed, idx, p):
    """float32 keep-scale of elements ``idx`` (numpy uint64 flat indices) under a resolved seed: 0 where dropped, else
    1 / (1 - p); p == 0 keeps everything at scale 1"""
    idx = np.asarray(idx, dtype=np.uint64)
    if p <= 0.0:
        return np.ones(idx.shape, dtype=np.float32)
    h = mix64(np.uint64((int(seed) * GOLDEN) & MASK64) + (idx >> np.uint64(2)))
    field = (h >> (np.uint64(16) * (idx & np.uint64(3)))) & np.uint64(0xFFFF)
    return np.where(field < np.uint64(threshold(p)), np.float32(0.0), inv_keep(p)).astype(np.float32)


def keep_scale_grid(seed, rows, cols, p, ld=None):
    """keep-scale of a [rows, cols] block whose element (r, c) uses index r * ld + c (ld defaults to cols)"""
    ld = cols if ld is None else ld
    idx = np.arange(rows, dtype=np.uint64)[:, None] * np.uint64(ld) + np.arange(cols, dtype=np.uint64)[None, :]
    return keep_scale(seed, idx, p)
