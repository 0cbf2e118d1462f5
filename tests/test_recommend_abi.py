"""CPU tests of the top-k recommendation entry points: nnr_topk_merge rejects bad arguments with NNR_ERR_ARG and a message
before any CUDA call (dummy pointers only), and CorpusScorer.recommend rejects bad inputs before any kernel launch."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NNR_ERR_ARG = -1
DUMMY = 256          # a non-NULL pointer that is never dereferenced: the checks run before any CUDA call


def _merge(k=10, T=100, B=4, lds=None, pos0=0, scores=DUMMY, best_score=DUMMY, best_pos=DUMMY, exclude=None,
           exclude_len=None, tile_ids=None, ldx=0):
    from nnr_b200 import _lib
    return _lib.lib.nnr_topk_merge(scores, T if lds is None else lds, B, T, pos0, tile_ids, exclude, exclude_len, ldx, k, 1,
                                   best_score, best_pos, None)


def _rejects(rc, what):
    from nnr_b200 import _lib
    msg = _lib.lib.nnr_last_error()
    assert rc == NNR_ERR_ARG, rc
    assert b'nnr_topk_merge' in msg and what.encode() in msg, msg


def test_topk_limits_match_the_header():
    from nnr_b200 import ops
    header = open(os.path.join(ROOT, 'include', 'nnr_b200.h')).read()
    for name, value in (('K', ops.TOPK_MAX_K), ('TILE', ops.TOPK_MAX_TILE), ('EXCLUDE', ops.TOPK_MAX_EXCLUDE)):
        assert int(re.search(r'#define\s+NNR_TOPK_MAX_%s\s+(\d+)' % name, header).group(1)) == value
    assert ops.TOPK_MAX_K >= 1024 and ops.TOPK_MAX_TILE >= 4096


@pytest.mark.parametrize('k', [0, -3, 1025])
def test_topk_merge_rejects_k_out_of_range(k):
    _rejects(_merge(k=k), 'k must be')


@pytest.mark.parametrize('T', [0, -1, 4097])
def test_topk_merge_rejects_tile_out_of_range(T):
    _rejects(_merge(T=T), 'T must be')


@pytest.mark.parametrize('which', ['scores', 'best_score', 'best_pos'])
def test_topk_merge_rejects_null_buffers(which):
    _rejects(_merge(**{which: None}), 'must not be NULL')


def test_topk_merge_rejects_bad_strides_positions_and_exclusion_lists():
    _rejects(_merge(T=100, lds=99), 'lds')
    _rejects(_merge(pos0=-1), 'pool positions')
    _rejects(_merge(pos0=2 ** 31 - 50, T=100), 'pool positions')
    _rejects(_merge(exclude=DUMMY, exclude_len=DUMMY, tile_ids=None, ldx=50), 'exclusion list needs')
    _rejects(_merge(exclude=DUMMY, exclude_len=None, tile_ids=DUMMY, ldx=50), 'exclusion list needs')
    _rejects(_merge(exclude=DUMMY, exclude_len=DUMMY, tile_ids=DUMMY, ldx=1025), 'ldx must be')


def test_topk_merge_with_no_rows_is_a_no_op():
    assert _merge(B=0) == 0


@pytest.fixture(scope='module')
def cpu_scorer():
    """a CorpusScorer of a tiny model on the CPU with a stand-in cache: enough to reach recommend()'s input checks"""
    import nnr_b200
    from nnr_b200.scoring import CorpusScorer
    from nnr_b200.synthetic import SyntheticMIND
    from oracle import nnr_oracle as O
    cfg = O.make_config(vocabulary_size=200, max_history_num=6, max_title_length=8, max_abstract_length=12,
                        subCategory_num=20, gcn_layer_num=1)
    syn = SyntheticMIND(news_num=40, vocabulary_size=200, subCategory_num=20, max_title_length=8, max_abstract_length=12,
                        max_history_num=6, lengths='uniform', seed=2)
    m = nnr_b200.Model(cfg)
    sc = CorpusScorer(m, syn.news_title_text, syn.news_title_mask, syn.news_abstract_text, syn.news_abstract_mask,
                      syn.news_category, syn.news_subCategory, chunk=16)
    hist, hl, _ = syn.sample_behaviors(3, news_num=2, seed=1)
    return sc, hist, hl, m.news_embedding_dim


def test_recommend_needs_encode_corpus_first(cpu_scorer):
    sc, hist, hl, D = cpu_scorer
    sc.cache = None
    with pytest.raises(RuntimeError, match='encode_corpus'):
        sc.recommend(hist, hl, torch.arange(10), 5)


@pytest.mark.parametrize('pool, k, what', [
    (np.arange(10), 0, 'k must be'),
    (np.arange(10), 1025, 'k must be'),
    (np.array([0, 5, 40]), 3, r'pool_ids must be in \[0, 40\)'),
    (np.array([-1, 5]), 3, r'pool_ids must be in \[0, 40\)'),
    (np.arange(10).reshape(2, 5), 3, '1-D integer'),
    (np.linspace(0, 1, 4), 3, '1-D integer'),
])
def test_recommend_rejects_bad_inputs_before_any_launch(cpu_scorer, pool, k, what):
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)          # stands in for encode_corpus(): only its shape is read before the checks pass
    before = ops.launch_count()
    with pytest.raises(ValueError, match=what):
        sc.recommend(hist, hl, pool, k)
    with pytest.raises(ValueError, match='pool_tile must be'):
        sc.recommend(hist, hl, np.arange(10), 3, pool_tile=4097)
    assert ops.launch_count() == before
