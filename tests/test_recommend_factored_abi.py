"""CPU tests of the factored cluster tail (recommend(exact=False)): nnr_cluster_tail_scores rejects bad arguments with its
error code and a message naming it, before any CUDA call (dummy pointers only), and recommend(exact=False) runs the same
input checks as the exact path before any kernel launch."""
import numpy as np
import pytest
import torch

from tests.test_recommend_abi import cpu_scorer  # noqa: F401  (fixture)

NNR_ERR_ARG, NNR_ERR_UNSUPPORTED = -1, -4
DUMMY = 256          # a 16-byte aligned non-NULL pointer that is never dereferenced: the checks run before any CUDA call
BUFFERS = ('Kp', 'g', 'Wg', 'idx', 'cmask', 'Qp', 'qk2', 'cand', 'bias', 'scores')


def _tail(B=4, H=50, Au=225, D=900, C1=19, T=100, lds=None, **ptr):
    from nnr_b200 import _lib
    p = {name: ptr.get(name, DUMMY) for name in BUFFERS}
    return _lib.lib.nnr_cluster_tail_scores(p['Kp'], p['g'], p['Wg'], p['idx'], p['cmask'], p['Qp'], p['qk2'], p['cand'],
                                            p['bias'], B, H, Au, D, C1, T, 0.1, p['scores'], T if lds is None else lds, None)


def _rejects(rc, code, what):
    from nnr_b200 import _lib
    msg = _lib.lib.nnr_last_error()
    assert rc == code, rc
    assert b'nnr_cluster_tail_scores' in msg and what.encode() in msg, msg


@pytest.mark.parametrize('which', BUFFERS)
def test_tail_rejects_null_buffers(which):
    _rejects(_tail(**{which: None}), NNR_ERR_ARG, 'must not be NULL')


@pytest.mark.parametrize('T', [0, -1, 4097])
def test_tail_rejects_tile_out_of_range(T):
    _rejects(_tail(T=T), NNR_ERR_ARG, 'T must be in [1, 4096]')


@pytest.mark.parametrize('H, C1', [(257, 19), (50, 73), (300, 100)])
def test_tail_rejects_more_slots_or_clusters_than_supported(H, C1):
    _rejects(_tail(H=H, C1=C1), NNR_ERR_UNSUPPORTED, 'H <= 256 and C1 <= 72')


@pytest.mark.parametrize('kw', [dict(B=-1), dict(H=0), dict(Au=0), dict(D=0), dict(C1=0)])
def test_tail_rejects_bad_sizes(kw):
    _rejects(_tail(**kw), NNR_ERR_ARG, 'bad sizes')


def test_tail_rejects_bad_strides_and_layouts():
    _rejects(_tail(T=100, lds=99), NNR_ERR_ARG, 'lds')
    _rejects(_tail(D=902), NNR_ERR_UNSUPPORTED, 'D % 4 == 0')
    _rejects(_tail(cand=DUMMY + 4), NNR_ERR_UNSUPPORTED, '16-byte aligned')


def test_tail_at_its_limits_and_with_no_users_is_a_no_op():
    assert _tail(B=0, H=256, C1=72, T=4096) == 0


def test_tail_is_a_dispatched_op():
    from nnr_b200 import ops
    assert 'cluster_tail_scores' in ops.DISPATCHED and hasattr(torch.ops.nnr, 'cluster_tail_scores')


@pytest.mark.parametrize('pool, k, what', [
    (np.arange(10), 0, 'k must be'),
    (np.arange(10), 1025, 'k must be'),
    (np.array([0, 5, 40]), 3, r'pool_ids must be in \[0, 40\)'),
    (np.arange(10).reshape(2, 5), 3, '1-D integer'),
])
def test_factored_recommend_rejects_bad_inputs_before_any_launch(cpu_scorer, pool, k, what):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)          # stands in for encode_corpus(): only its shape is read before the checks pass
    before = ops.launch_count()
    with pytest.raises(ValueError, match=what):
        sc.recommend(hist, hl, pool, k, exact=False)
    with pytest.raises(ValueError, match='pool_tile must be'):
        sc.recommend(hist, hl, np.arange(10), 3, pool_tile=4097, exact=False)
    with pytest.raises(ValueError, match='max_per_category must be'):
        sc.recommend(hist, hl, np.arange(10), 3, max_per_category=0, exact=False)
    with pytest.raises(ValueError, match='collective=True needs'):
        sc.recommend(hist, hl, np.arange(10), 3, collective=True, exact=False)
    assert ops.launch_count() == before


def test_factored_recommend_default_tile_is_the_pool_up_to_the_tile_limit(cpu_scorer):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)
    for P, want in ((1, 1), (37, 37)):
        assert sc._recommend_inputs(hist, hl, np.arange(P), 3, True, None, None, exact=False)[4] == want
    assert sc._recommend_inputs(hist, hl, np.zeros(5000, dtype=np.int64), 3, True, None, None, exact=False)[4] == ops.TOPK_MAX_TILE
    assert sc._recommend_inputs(hist, hl, np.arange(37), 3, True, None, None)[4] == sc.default_pool_tile(len(hl))


def test_exact_is_part_of_the_collective_agreement():
    from nnr_b200.scoring import CorpusScorer
    assert 'exact' in CorpusScorer._FIELDS
