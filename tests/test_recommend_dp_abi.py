"""CPU tests of the data-parallel top-k recommendation: nnr_topk_merge_lists and nnr_topk_merge_lists_capped reject bad
arguments with NNR_ERR_ARG and a message naming the entry point before any CUDA call (dummy pointers only), and
CorpusScorer.recommend(collective=True) without a process group raises ValueError."""
import numpy as np
import pytest
import torch

from tests.test_recommend_abi import cpu_scorer  # noqa: F401  (fixture)

NNR_ERR_ARG = -1
DUMMY = 256          # a non-NULL pointer that is never dereferenced: the checks run before any CUDA call


def _merge(k=10, T=10, B=4, lds=None, pos=DUMMY, ldp=None, scores=DUMMY, best_score=DUMMY, best_pos=DUMMY):
    from nnr_b200 import _lib
    return _lib.lib.nnr_topk_merge_lists(scores, T if lds is None else lds, B, T, pos, T if ldp is None else ldp, k, 1,
                                         best_score, best_pos, None)


def _merge_capped(k=10, T=10, B=4, lds=None, pos=DUMMY, ldp=None, grp=DUMMY, ldg=None, num_groups=18, cap=2,
                  scores=DUMMY, best_score=DUMMY, best_pos=DUMMY, best_group=DUMMY):
    from nnr_b200 import _lib
    return _lib.lib.nnr_topk_merge_lists_capped(scores, T if lds is None else lds, B, T, pos, T if ldp is None else ldp, grp,
                                                T if ldg is None else ldg, num_groups, cap, k, 1, best_score, best_pos,
                                                best_group, None)


def _rejects(rc, who, what):
    from nnr_b200 import _lib
    msg = _lib.lib.nnr_last_error()
    assert rc == NNR_ERR_ARG, rc
    assert who.encode() + b':' in msg and what.encode() in msg, msg


@pytest.mark.parametrize('merge, who', [(_merge, 'nnr_topk_merge_lists'), (_merge_capped, 'nnr_topk_merge_lists_capped')])
def test_list_merges_reject_what_the_tile_merge_rejects(merge, who):
    for k in (0, -3, 1025):
        _rejects(merge(k=k), who, 'k must be')
    for T in (0, -1, 4097):
        _rejects(merge(T=T, lds=4097, ldp=4097, **({'ldg': 4097} if merge is _merge_capped else {})), who, 'T must be')
    _rejects(merge(B=-1), who, 'B must be')
    _rejects(merge(T=100, lds=99, ldp=100, **({'ldg': 100} if merge is _merge_capped else {})), who, 'lds')
    for which in ('scores', 'best_score', 'best_pos'):
        _rejects(merge(**{which: None}), who, 'must not be NULL')
    _rejects(merge(pos=None), who, 'pos must not be NULL')
    _rejects(merge(T=100, ldp=99, lds=100, **({'ldg': 100} if merge is _merge_capped else {})), who, 'ldp (99) < T (100)')


def test_capped_list_merge_rejects_bad_groups():
    who = 'nnr_topk_merge_lists_capped'
    _rejects(_merge_capped(grp=None), who, 'grp and best_group must not be NULL')
    _rejects(_merge_capped(best_group=None), who, 'grp and best_group must not be NULL')
    _rejects(_merge_capped(T=100, ldg=99, lds=100, ldp=100), who, 'ldg (99) < T (100)')
    for cap in (0, -1):
        _rejects(_merge_capped(cap=cap), who, 'cap must be >= 1')
    for num_groups in (0, -5, 1025):
        _rejects(_merge_capped(num_groups=num_groups), who, 'num_groups must be in [1, 1024]')


def test_list_merges_accept_the_largest_list_and_no_rows():
    """a k = 1024 best list is one launch (T = k); B = 0 returns before any CUDA call"""
    assert _merge(B=0, k=1024, T=1024) == 0
    assert _merge_capped(B=0, k=1024, T=1024, num_groups=1024, cap=1) == 0
    assert _merge(B=0, k=1, T=4096, ldp=5000) == 0


def test_collective_recommend_needs_a_process_group(cpu_scorer):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)
    before = ops.launch_count()
    with pytest.raises(ValueError, match='collective=True needs a scorer built with a process_group'):
        sc.recommend(hist, hl, np.arange(10), 5, collective=True)
    assert ops.launch_count() == before
