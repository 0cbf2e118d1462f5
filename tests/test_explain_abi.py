"""CPU tests of score explanations (CorpusScorer.explain): nnr_cluster_tail_explain_packed rejects bad arguments with the
error codes and messages of nnr_cluster_tail_scores_packed before any CUDA call (dummy pointers only), explain() checks
its arguments before any kernel launch, and tests.explain_ref.sue_explain splits oracle.sue_forward's click score exactly
(fp64)."""
import numpy as np
import pytest
import torch

from tests.test_evaluate_factored_abi import DUMMY, NNR_ERR_ARG, NNR_ERR_UNSUPPORTED, _impressions
from tests.test_recommend_abi import cpu_scorer  # noqa: F401  (fixture)

BUFFERS = ('Kp', 'g', 'Wg', 'idx', 'cmask', 'row_off', 'Qp', 'qk2', 'cand', 'bias', 'scores', 'alpha_out', 'beta_out',
           'contrib_out')


def _explain(B=4, H=50, Au=225, D=900, C1=19, n_max=300, rows=1200, lds=None, **ptr):
    from nnr_b200 import _lib
    p = {name: ptr.get(name, DUMMY) for name in BUFFERS}
    return _lib.lib.nnr_cluster_tail_explain_packed(p['Kp'], p['g'], p['Wg'], p['idx'], p['cmask'], p['row_off'], rows,
                                                    p['Qp'], p['qk2'], p['cand'], p['bias'], B, H, Au, D, C1, n_max, 0.1,
                                                    p['scores'], n_max if lds is None else lds, p['alpha_out'],
                                                    p['beta_out'], p['contrib_out'], None)


def _rejects(rc, code, what):
    from nnr_b200 import _lib
    msg = _lib.lib.nnr_last_error()
    assert rc == code, rc
    assert b'nnr_cluster_tail_explain_packed' in msg and what.encode() in msg, msg


@pytest.mark.parametrize('which', BUFFERS)
def test_explain_rejects_null_buffers(which):
    _rejects(_explain(**{which: None}), NNR_ERR_ARG, 'must not be NULL')


@pytest.mark.parametrize('kw', [dict(B=-1), dict(H=0), dict(Au=0), dict(D=0), dict(C1=0), dict(B=2 ** 30, n_max=300)])
def test_explain_rejects_bad_sizes(kw):
    _rejects(_explain(**kw), NNR_ERR_ARG, 'bad sizes')


@pytest.mark.parametrize('n_max, lds', [(0, 300), (-1, 300), (301, 300)])
def test_explain_rejects_n_max_outside_one_to_lds(n_max, lds):
    _rejects(_explain(n_max=n_max, lds=lds), NNR_ERR_ARG, 'n_max must be in [1, lds')


@pytest.mark.parametrize('rows', [-1, 2 ** 31, 2 ** 40])
def test_explain_rejects_bad_rows(rows):
    _rejects(_explain(rows=rows), NNR_ERR_ARG, 'rows must be in [0, 2^31)')


@pytest.mark.parametrize('H, C1', [(257, 19), (50, 73), (300, 100)])
def test_explain_rejects_more_slots_or_clusters_than_supported(H, C1):
    _rejects(_explain(H=H, C1=C1), NNR_ERR_UNSUPPORTED, 'H <= 256 and C1 <= 72')


@pytest.mark.parametrize('which', ['g', 'Wg', 'qk2', 'cand', 'bias'])
def test_explain_rejects_misaligned_buffers(which):
    _rejects(_explain(**{which: DUMMY + 4}), NNR_ERR_UNSUPPORTED, '16-byte aligned')


def test_explain_rejects_d_not_a_multiple_of_4():
    _rejects(_explain(D=902), NNR_ERR_UNSUPPORTED, 'D % 4 == 0')


def test_explain_at_its_limits_and_with_no_users_is_a_no_op():
    assert _explain(B=0, H=256, C1=72, n_max=300, rows=0) == 0
    assert _explain(B=0, n_max=1, lds=1, rows=2 ** 31 - 1) == 0


def test_explain_is_a_dispatched_op():
    from nnr_b200 import ops
    assert 'cluster_tail_explain_packed' in ops.DISPATCHED and hasattr(torch.ops.nnr, 'cluster_tail_explain_packed')


# ---- CorpusScorer.explain(): argument checks -------------------------------------------------------------------------
def test_explain_needs_encode_corpus_first(cpu_scorer):  # noqa: F811
    sc, hist, hl, D = cpu_scorer
    sc.cache = None
    with pytest.raises(RuntimeError, match='CorpusScorer.explain: call encode_corpus'):
        sc.explain(hist, hl, np.ones((3, 2), dtype=np.int64))


@pytest.mark.parametrize('exact', [False, True])
@pytest.mark.parametrize('edit, what', [
    (lambda c, n: (c, np.array([5, 6, 0])), r'candidate_count must be in \[0, 5\]'),
    (lambda c, n: (c, np.array([5, -1, 0])), r'candidate_count must be in \[0, 5\]'),
    (lambda c, n: (c, np.array([5, 2])), r'candidate_count must be an integer tensor of shape \[3\]'),
    (lambda c, n: (c, np.array([5.0, 2.0, 0.0])), r'candidate_count must be an integer tensor of shape \[3\]'),
    (lambda c, n: (np.where(np.arange(5) == 1, 40, c), n), r'valid candidate ids must be in \[0, 40\)'),
    (lambda c, n: (np.where(np.arange(5) == 0, -1, c), n), r'valid candidate ids must be in \[0, 40\)'),
    (lambda c, n: (c[0], None), '2-D integer'),
    (lambda c, n: (c.astype(np.float32), None), '2-D integer'),
])
def test_explain_rejects_bad_arguments_before_any_launch(cpu_scorer, edit, what, exact):  # noqa: F811
    from nnr_b200 import ops
    sc, hist, hl, D = cpu_scorer
    sc.cache = torch.zeros(40, D)          # stands in for encode_corpus(): only its shape is read before the checks pass
    cand, cnt, _ = _impressions()
    cand, cnt = edit(cand, cnt)
    before = ops.launch_count()
    with pytest.raises(ValueError, match='CorpusScorer.explain: .*' + what):
        sc.explain(hist, hl, cand, cnt, exact=exact)
    assert ops.launch_count() == before


# ---- explain_ref.sue_explain against oracle.sue_forward, fp64 -------------------------------------------------------
def _oracle_inputs(user_encoder, B=5, H=8, n=6, seed=0):
    from oracle import graph as OG
    from oracle import nnr_oracle as O
    cfg = O.make_config(user_encoder=user_encoder, hidden_dim=16, attention_dim=12, category_embedding_dim=8,
                        subCategory_embedding_dim=8, max_history_num=H, gcn_layer_num=2, category_num=6)
    p = O.formula_params(cfg, dtype=torch.float64)
    D = p['user_encoder.proxy_node_embedding' if user_encoder != 'SUE_wo_GCN' else 'user_encoder.intraCluster_Q.weight'].shape[1]
    rng = np.random.default_rng(seed)
    lens = [H, 3, 1, 0, 5][:B]
    g, cm, ci = zip(*[OG.build_history_graph(rng.integers(0, 6, L), H, 6) for L in lens])
    gen = torch.Generator().manual_seed(seed)
    hist = torch.randn(B, H, D, generator=gen, dtype=torch.float64)
    cand = torch.randn(B, n, D, generator=gen, dtype=torch.float64)
    t = lambda x: torch.from_numpy(np.stack(x))
    return p, cfg, hist, t(g).double(), t(cm), t(ci), cand


@pytest.mark.parametrize('user_encoder', ['SUE', 'SUE_wo_GCN', 'SUE_wo_HCA'])
def test_reference_explain_splits_sue_forward_exactly(user_encoder):
    from oracle import nnr_oracle as O
    from tests.explain_ref import sue_explain
    p, cfg, hist, graph, cmask, cidx, cand = _oracle_inputs(user_encoder)
    alpha, beta, fc, user = sue_explain(p, cfg, hist, graph, cmask, cidx, cand)
    ref = O.sue_forward(p, cfg, hist, graph, cmask.clone(), cidx, cand)
    assert torch.allclose(user, ref, rtol=0, atol=1e-12)
    B, n, H = alpha.shape
    if beta is None:                                                                   # SUE_wo_HCA: no clusters
        assert torch.allclose(alpha.sum(2), torch.ones(B, n, dtype=alpha.dtype), rtol=0, atol=1e-12)
        return
    score = (user * cand).sum(2)
    assert torch.allclose((beta * fc).sum(2), score, rtol=0, atol=1e-12)
    assert torch.allclose(beta.sum(2), torch.ones(B, n, dtype=beta.dtype), rtol=0, atol=1e-12)
    cm = cmask.clone()
    cm[:, -1] = True
    assert (beta.masked_select(~cm[:, None, :].expand_as(beta)) == 0).all()          # masked clusters weigh nothing
    for b in range(B):                                                                 # alpha sums to 1 in every cluster
        for c in cidx[b].unique().tolist():
            assert torch.allclose(alpha[b][:, cidx[b] == c].sum(1), torch.ones(n, dtype=alpha.dtype), rtol=0, atol=1e-12)
