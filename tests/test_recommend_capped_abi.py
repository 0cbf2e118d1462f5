"""CPU tests of the per-category cap of top-k recommendation: nnr_topk_merge_capped rejects bad arguments with NNR_ERR_ARG
and a message naming itself before any CUDA call (dummy pointers only), and CorpusScorer.recommend(max_per_category=)
rejects a bad cap or out-of-range corpus categories before any kernel launch."""
import os
import re

import numpy as np
import pytest
import torch

from tests.test_recommend_abi import cpu_scorer  # noqa: F401  (fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NNR_ERR_ARG = -1
DUMMY = 256          # a non-NULL pointer that is never dereferenced: the checks run before any CUDA call


def _merge(k=10, T=100, B=4, lds=None, pos0=0, scores=DUMMY, best_score=DUMMY, best_pos=DUMMY, exclude=None,
           exclude_len=None, tile_ids=DUMMY, ldx=0, id_group=DUMMY, num_groups=18, cap=2, best_group=DUMMY):
    from nnr_b200 import _lib
    return _lib.lib.nnr_topk_merge_capped(scores, T if lds is None else lds, B, T, pos0, tile_ids, exclude, exclude_len, ldx,
                                          k, 1, id_group, num_groups, cap, best_score, best_pos, best_group, None)


def _rejects(rc, what):
    from nnr_b200 import _lib
    msg = _lib.lib.nnr_last_error()
    assert rc == NNR_ERR_ARG, rc
    assert b'nnr_topk_merge_capped' in msg and what.encode() in msg, msg


def test_topk_max_groups_matches_the_header():
    from nnr_b200 import ops
    header = open(os.path.join(ROOT, 'include', 'nnr_b200.h')).read()
    assert int(re.search(r'#define\s+NNR_TOPK_MAX_GROUPS\s+(\d+)', header).group(1)) == ops.TOPK_MAX_GROUPS == 1024


@pytest.mark.parametrize('k', [0, -3, 1025])
def test_capped_merge_rejects_k_out_of_range(k):
    _rejects(_merge(k=k), 'k must be')


@pytest.mark.parametrize('T', [0, -1, 4097])
def test_capped_merge_rejects_tile_out_of_range(T):
    _rejects(_merge(T=T), 'T must be')


@pytest.mark.parametrize('which', ['scores', 'best_score', 'best_pos'])
def test_capped_merge_rejects_null_buffers(which):
    _rejects(_merge(**{which: None}), 'must not be NULL')


@pytest.mark.parametrize('which', ['id_group', 'best_group', 'tile_ids'])
def test_capped_merge_rejects_null_group_buffers(which):
    _rejects(_merge(**{which: None}), 'id_group, best_group and tile_ids must not be NULL')


def test_capped_merge_rejects_what_the_uncapped_merge_rejects():
    _rejects(_merge(B=-1), 'B must be')
    _rejects(_merge(T=100, lds=99), 'lds')
    _rejects(_merge(pos0=-1), 'pool positions')
    _rejects(_merge(pos0=2 ** 31 - 50, T=100), 'pool positions')
    _rejects(_merge(exclude=DUMMY, exclude_len=None, ldx=50), 'exclusion list needs')
    _rejects(_merge(exclude=DUMMY, exclude_len=DUMMY, ldx=1025), 'ldx must be')


@pytest.mark.parametrize('cap', [0, -1])
def test_capped_merge_rejects_a_cap_below_one(cap):
    _rejects(_merge(cap=cap), 'cap must be >= 1')


@pytest.mark.parametrize('num_groups', [0, -5, 1025])
def test_capped_merge_rejects_num_groups_out_of_range(num_groups):
    _rejects(_merge(num_groups=num_groups), 'num_groups must be in [1, 1024]')


def test_capped_merge_with_no_rows_is_a_no_op():
    assert _merge(B=0) == 0
    assert _merge(B=0, num_groups=1024, cap=1) == 0


@pytest.mark.parametrize('m', [0, -2, 1.0, 2.5, '3', True, False, np.float32(2), torch.tensor(2)])
def test_recommend_rejects_a_bad_max_per_category_before_any_launch(cpu_scorer, m):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)          # stands in for encode_corpus(): only its shape is read before the checks pass
    before = ops.launch_count()
    with pytest.raises(ValueError, match='max_per_category must be'):
        sc.recommend(hist, hl, np.arange(10), 5, max_per_category=m)
    assert ops.launch_count() == before


@pytest.mark.parametrize('bad', [-1, 1024, 5000])
def test_recommend_rejects_out_of_range_categories_before_any_launch(cpu_scorer, bad):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)
    cat = sc.cat
    try:
        sc.cat = cat.clone()
        sc.cat[7] = bad
        sc._num_groups = None
        before = ops.launch_count()
        with pytest.raises(ValueError, match=r'category ids in \[0, 1024\)'):
            sc.recommend(hist, hl, np.arange(10), 5, max_per_category=2)
        with pytest.raises(ValueError, match=r'category ids in \[0, 1024\)'):     # checked again until it passes
            sc.recommend(hist, hl, np.arange(10), 5, max_per_category=1)
        assert ops.launch_count() == before
    finally:
        sc.cat = cat
        sc._num_groups = None


def test_uncapped_calls_do_not_check_the_categories(cpu_scorer):  # noqa: F811
    """max_per_category None or >= k takes the uncapped path, which reads no category: a bad id does not stop it (it
    gets as far as the CPU scorer's first kernel, which cannot run on CPU tensors)"""
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)
    cat = sc.cat
    try:
        sc.cat = cat.clone()
        sc.cat[7] = 5000
        sc._num_groups = None
        for m in (None, 5, 9):
            with pytest.raises(Exception) as e:
                sc.recommend(hist, hl, np.arange(10), 5, max_per_category=m)
            assert not isinstance(e.value, ValueError), e.value
        assert sc._num_groups is None
    finally:
        sc.cat = cat
        sc._num_groups = None


def test_recommend_counts_the_groups_once_per_scorer(cpu_scorer):  # noqa: F811
    sc, hist, hl, D = cpu_scorer
    sc._num_groups = None
    want = int(sc.cat.max()) + 1
    assert sc._category_groups() == want
    cat = sc.cat
    try:
        sc.cat = cat.clone()
        sc.cat[0] = -1                       # not looked at again once the check has passed
        assert sc._category_groups() == want
    finally:
        sc.cat = cat
        sc._num_groups = None
