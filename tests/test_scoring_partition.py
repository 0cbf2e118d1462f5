"""CPU test of the contiguous partition that shares corpus chunks / impression batches between the ranks of a sharded
``CorpusScorer``."""
import pytest

from nnr_b200.scoring import contiguous_blocks


@pytest.mark.parametrize('block', [1, 64, 256])
@pytest.mark.parametrize('world', [1, 2, 3, 4, 8])
@pytest.mark.parametrize('nitems', [0, 1, 44, 63, 64, 65, 150, 300, 1000, 16384, 100000])
def test_contiguous_blocks_cover_every_item_once(nitems, world, block):
    nblocks = -(-nitems // block)
    k, parts = contiguous_blocks(nblocks, world)
    assert len(parts) == world
    assert k * world >= nblocks and (k - 1) * world < max(nblocks, 1)        # k = ceil(nblocks / world)
    seen = []
    for first, end in parts:
        assert 0 <= first <= end <= nblocks
        assert end - first <= k                                              # no rank holds more than the balanced maximum
        lo, hi = min(first * block, nitems), min(end * block, nitems)        # items of the rank: boundaries on block multiples
        assert lo % block == 0 or lo == nitems
        assert hi % block == 0 or hi == nitems
        seen.extend(range(lo, hi))
    assert seen == list(range(nitems))                                       # every item exactly once, in rank order
    counts = [end - first for first, end in parts]
    full = [c for c in counts if c]
    assert all(c == k for c in full[:-1])                                    # rank r's k-block send buffer starts at r*k blocks
    # the ranks that own blocks hold k except the last, which may hold fewer; the ranks after it own none
    assert counts == full + [0] * (world - len(full))


def test_contiguous_blocks_examples():
    assert contiguous_blocks(5, 2) == (3, [(0, 3), (3, 5)])
    assert contiguous_blocks(5, 4) == (2, [(0, 2), (2, 4), (4, 5), (5, 5)])
    assert contiguous_blocks(2, 4) == (1, [(0, 1), (1, 2), (2, 2), (2, 2)])   # fewer blocks than ranks: idle ranks
    assert contiguous_blocks(64, 8) == (8, [(8 * r, 8 * r + 8) for r in range(8)])
    assert contiguous_blocks(0, 3) == (0, [(0, 0)] * 3)
