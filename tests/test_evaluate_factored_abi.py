"""CPU tests of evaluation through the factored cluster tail (score / evaluate(exact=False)): nnr_cluster_tail_scores_packed
rejects bad arguments with its error code and a message naming it, before any CUDA call (dummy pointers only), and
score(exact=False) / evaluate(exact=False) check the counts and the valid candidate ids before any kernel launch."""
import numpy as np
import pytest
import torch

from tests.test_recommend_abi import cpu_scorer  # noqa: F401  (fixture)

NNR_ERR_ARG, NNR_ERR_UNSUPPORTED = -1, -4
DUMMY = 256          # a 16-byte aligned non-NULL pointer that is never dereferenced: the checks run before any CUDA call
BUFFERS = ('Kp', 'g', 'Wg', 'idx', 'cmask', 'row_off', 'Qp', 'qk2', 'cand', 'bias', 'scores')


def _packed(B=4, H=50, Au=225, D=900, C1=19, n_max=300, rows=1200, lds=None, **ptr):
    from nnr_b200 import _lib
    p = {name: ptr.get(name, DUMMY) for name in BUFFERS}
    return _lib.lib.nnr_cluster_tail_scores_packed(p['Kp'], p['g'], p['Wg'], p['idx'], p['cmask'], p['row_off'], rows,
                                                   p['Qp'], p['qk2'], p['cand'], p['bias'], B, H, Au, D, C1, n_max, 0.1,
                                                   p['scores'], n_max if lds is None else lds, None)


def _rejects(rc, code, what):
    from nnr_b200 import _lib
    msg = _lib.lib.nnr_last_error()
    assert rc == code, rc
    assert b'nnr_cluster_tail_scores_packed' in msg and what.encode() in msg, msg


@pytest.mark.parametrize('which', BUFFERS)
def test_packed_rejects_null_buffers(which):
    _rejects(_packed(**{which: None}), NNR_ERR_ARG, 'must not be NULL')


@pytest.mark.parametrize('kw', [dict(B=-1), dict(H=0), dict(Au=0), dict(D=0), dict(C1=0), dict(B=2 ** 30, n_max=300)])
def test_packed_rejects_bad_sizes(kw):
    _rejects(_packed(**kw), NNR_ERR_ARG, 'bad sizes')


@pytest.mark.parametrize('n_max, lds', [(0, 300), (-1, 300), (301, 300)])
def test_packed_rejects_n_max_outside_one_to_lds(n_max, lds):
    _rejects(_packed(n_max=n_max, lds=lds), NNR_ERR_ARG, 'n_max must be in [1, lds')


@pytest.mark.parametrize('rows', [-1, 2 ** 31, 2 ** 40])
def test_packed_rejects_bad_rows(rows):
    _rejects(_packed(rows=rows), NNR_ERR_ARG, 'rows must be in [0, 2^31)')


@pytest.mark.parametrize('H, C1', [(257, 19), (50, 73), (300, 100)])
def test_packed_rejects_more_slots_or_clusters_than_supported(H, C1):
    _rejects(_packed(H=H, C1=C1), NNR_ERR_UNSUPPORTED, 'H <= 256 and C1 <= 72')


@pytest.mark.parametrize('which', ['g', 'Wg', 'qk2', 'cand', 'bias'])
def test_packed_rejects_misaligned_buffers(which):
    _rejects(_packed(**{which: DUMMY + 4}), NNR_ERR_UNSUPPORTED, '16-byte aligned')


def test_packed_rejects_d_not_a_multiple_of_4():
    _rejects(_packed(D=902), NNR_ERR_UNSUPPORTED, 'D % 4 == 0')


def test_packed_at_its_limits_and_with_no_users_is_a_no_op():
    assert _packed(B=0, H=256, C1=72, n_max=300, rows=0) == 0
    assert _packed(B=0, n_max=1, lds=1, rows=2 ** 31 - 1) == 0


def test_packed_is_a_dispatched_op():
    from nnr_b200 import ops
    assert 'cluster_tail_scores_packed' in ops.DISPATCHED and hasattr(torch.ops.nnr, 'cluster_tail_scores_packed')


def _impressions(n_imp=3, n_max=5):
    cand = np.tile(np.arange(1, n_max + 1), (n_imp, 1))
    cnt = np.array([n_max, 2, 0][:n_imp] + [1] * max(0, n_imp - 3))
    lab = np.zeros((n_imp, n_max), dtype=np.int64)
    lab[:, 0] = 1
    return cand, cnt, lab


@pytest.mark.parametrize('edit, what', [
    (lambda c, n: (c, np.array([5, 6, 0])), r'candidate_count must be in \[0, 5\]'),
    (lambda c, n: (c, np.array([5, -1, 0])), r'candidate_count must be in \[0, 5\]'),
    (lambda c, n: (c, np.array([5, 2])), r'candidate_count must be an integer tensor of shape \[3\]'),
    (lambda c, n: (c, np.array([[5, 2, 0]])), r'candidate_count must be an integer tensor of shape \[3\]'),
    (lambda c, n: (np.where(np.arange(5) == 1, 40, c), n), r'valid candidate ids must be in \[0, 40\)'),
    (lambda c, n: (np.where(np.arange(5) == 0, -1, c), n), r'valid candidate ids must be in \[0, 40\)'),
])
def test_factored_evaluate_rejects_bad_counts_and_ids_before_any_launch(cpu_scorer, edit, what):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)          # stands in for encode_corpus(): only its shape is read before the checks pass
    cand, cnt, lab = _impressions()
    cand, cnt = edit(cand, cnt)
    before = ops.launch_count()
    with pytest.raises(ValueError, match=what):
        sc.evaluate(hist, hl, cand, cnt, lab, exact=False)
    assert ops.launch_count() == before


def test_factored_evaluate_does_not_read_padding_ids(cpu_scorer):  # noqa: F811
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)
    cand, cnt, _ = _impressions()
    cand = np.where(np.arange(5)[None, :] < cnt[:, None], cand, -1)          # padding may be anything: -1 passes the checks
    cid, c = sc._packed_inputs('evaluate', cand, cnt)
    assert torch.equal(cid, torch.as_tensor(cand)) and c.tolist() == cnt.tolist()


@pytest.mark.parametrize('cand, what', [
    (np.array([[1, 2], [3, 40], [5, 6]]), r'valid candidate ids must be in \[0, 40\)'),
    (np.array([[1, 2], [-1, 4], [5, 6]]), r'valid candidate ids must be in \[0, 40\)'),
    (np.array([1, 2, 3]), '2-D integer'),
    (np.ones((3, 2)), '2-D integer'),
])
def test_factored_score_rejects_out_of_range_ids_before_any_launch(cpu_scorer, cand, what):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)
    before = ops.launch_count()
    with pytest.raises(ValueError, match=what):
        sc.score(hist, hl, cand, exact=False)
    assert ops.launch_count() == before
