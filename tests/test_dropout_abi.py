"""CPU checks of the host dropout reference (tests/dropout_ref.py) that the GPU tests pin every mask against."""
import numpy as np
import pytest

from tests import dropout_ref as R


def _keep_scale_int(seed, i, p):
    """one element, straight from the rule in Python ints"""
    h = R.mix64_int(((seed * R.GOLDEN) & R.MASK64) + (i >> 2))
    field = (h >> (16 * (i & 3))) & 0xFFFF
    thr = int(np.float32(p) * np.float32(65536.0))
    return 0.0 if field < thr else float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def test_mix64_matches_int_definition():
    rng = np.random.default_rng(0)
    xs = np.concatenate([rng.integers(0, 2 ** 63, 500, dtype=np.uint64) * np.uint64(2) + np.uint64(1),
                         np.array([0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 62 - 1, 2 ** 64 - 1], dtype=np.uint64)])
    got = R.mix64(xs)
    assert [int(v) for v in got] == [R.mix64_int(int(x)) for x in xs]
    # a fixed value, so a change to the constants cannot pass unnoticed
    assert R.mix64_int(1) == 0xB456BCFC34C2CB2C


@pytest.mark.parametrize('seed', [0, 1, 0x2F3A5C7E9B1D4F61, 2 ** 62 - 1, 2 ** 62 - 2])
@pytest.mark.parametrize('p', [0.1, 0.25, 0.9])
def test_keep_scale_matches_scalar_rule(seed, p):
    rng = np.random.default_rng(seed % 1000 + int(p * 100))
    idx = np.concatenate([rng.integers(0, 2 ** 20, 300, dtype=np.uint64), rng.integers(2 ** 32 - 8, 2 ** 32 + 8, 50, dtype=np.uint64),
                          rng.integers(2 ** 32, 2 ** 63, 300, dtype=np.uint64)])
    got = R.keep_scale(seed, idx, p)
    assert got.dtype == np.float32
    ref = np.array([_keep_scale_int(seed, int(i), p) for i in idx], dtype=np.float32)
    assert np.array_equal(got, ref)


def test_one_hash_per_aligned_quad():
    """indices 4q .. 4q+3 are the four 16-bit fields of one hash, lowest field first"""
    seed, p = 0x2F3A5C7E9B1D4F61, 0.5
    thr = R.threshold(p)
    for q in (0, 1, 12345, 2 ** 40 + 7):
        h = R.mix64_int(((seed * R.GOLDEN) & R.MASK64) + q)
        fields = [(h >> (16 * k)) & 0xFFFF for k in range(4)]
        want = np.array([0.0 if f < thr else 2.0 for f in fields], dtype=np.float32)
        got = R.keep_scale(seed, np.arange(4 * q, 4 * q + 4, dtype=np.uint64), p)
        assert np.array_equal(got, want), q
    # the grid helper indexes r * ld + c
    g = R.keep_scale_grid(seed, 5, 7, 0.3, ld=9)
    flat = R.keep_scale(seed, (np.arange(5)[:, None] * 9 + np.arange(7)[None, :]).astype(np.uint64), 0.3)
    assert np.array_equal(g, flat)


def test_tiny_p_drops_nothing_but_still_scales():
    p = 1e-6
    assert R.threshold(p) == 0
    s = R.keep_scale(7, np.arange(100000, dtype=np.uint64), p)
    assert np.all(s == np.float32(1.0) / (np.float32(1.0) - np.float32(p)))
    assert np.all(s > 1.0)
    assert np.all(R.keep_scale(7, np.arange(100, dtype=np.uint64), 0.0) == 1.0)


@pytest.mark.parametrize('p', [0.1, 0.2, 0.5, 0.9])
def test_keep_fraction(p):
    n = 1 << 20
    s = R.keep_scale(0x2F3A5C7E9B1D4F61, np.arange(n, dtype=np.uint64), p)
    keep = (s != 0).mean()
    q = 1.0 - R.threshold(p) / 65536.0
    assert abs(keep - (1.0 - p)) < 3.0 * np.sqrt(p * (1.0 - p) / n) + abs(q - (1.0 - p))
    assert np.all(s[s != 0] == R.inv_keep(p))


def test_indirect_seed_resolution():
    base, site = 0x123456789ABCDEF0, 5
    x = (base + site * 0x9E3779B97F4A7C15) % 2 ** 64
    x ^= x >> 33
    x = x * 0xFF51AFD7ED558CCD % 2 ** 64
    x ^= x >> 33
    x = x * 0xC4CEB9FE1A85EC53 % 2 ** 64
    x ^= x >> 33
    assert R.resolve_indirect(base, site) == x >> 2 < 2 ** 62
    ptr = 0x00007F0012345670                                  # bits 0..47: the base's device address
    seed = R.INDIRECT | (site << 48) | ptr
    assert R.resolve_seed(seed, base) == x >> 2
    # site bits 48..61 only; the address does not enter the hash
    assert R.resolve_seed(R.INDIRECT | (0x3FFF << 48) | 0xFFFFFFFFFFFF, base) == R.resolve_indirect(base, 0x3FFF)
    # a base near 2^64 wraps
    assert R.resolve_indirect(2 ** 64 - 1, 1) == R.mix64_int((2 ** 64 - 1 + R.GOLDEN) % 2 ** 64) >> 2
    # direct seeds (< 2^62) are used as they are
    assert R.resolve_seed(2 ** 62 - 1) == 2 ** 62 - 1 and R.resolve_seed(0) == 0
