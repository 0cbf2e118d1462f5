"""GPU tests of score explanations (CorpusScorer.explain, nnr_cluster_tail_explain_packed).

  * the explain kernel against a float64 reference of alpha, beta and beta * (f . cand): counts 0, ragged and above 64,
    H = 256 with C1 = 72 (the 2-warp CTA), D % 8 == 4; its scores equal nnr_cluster_tail_scores_packed's bit for bit,
    and nothing is written past a count or outside a tensor;
  * explain(exact=True / False) against tests.explain_ref.sue_explain for SUE, SUE_wo_GCN, SUE_wo_HCA and a non-default
    graph flag; the scores equal score()'s bit for bit, the two paths agree, the cluster terms sum to the score, masked
    clusters weigh exactly 0;
  * ragged lists: padding ids are never read, outputs past the counts are 0, the padding width does not matter;
  * deterministic, graph replay equals host launches;
  * the explanation of a recommend() result, fill entries included.
"""
import math

import numpy as np
import pytest
import torch

from oracle import nnr_oracle as O
from tests.explain_ref import sue_explain
from tests.test_evaluate_factored_gpu import _packed_inputs, _ragged
from tests.test_recommend_gpu import (CHUNK, H, NEWS, TOL, _build, _config, _corpus, _scorer,
                                      sue)  # noqa: F401  (sue: fixture)
from tests.util import rel_err

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.contiguous().cpu().view(torch.int32)


# ---- the kernel alone --------------------------------------------------------------------------------------------------
def _reference(Kp, g, W, idx, cmask, Qp, qk2, cand, bias, scale):
    """float64, unfactored, for one user: (alpha [T, H] in history order, beta [T, C1], beta * (f . cand) [T, C1])"""
    C1 = cmask.shape[1]
    onehot = torch.nn.functional.one_hot(idx[0].clamp(0, C1 - 1), C1).to(torch.float64)         # [H, C1]
    s = scale * Qp @ Kp[0].T                                                                      # [T, H]
    same = onehot @ onehot.T
    m = torch.where(same[None] > 0, s[:, None, :], torch.tensor(-math.inf, dtype=s.dtype, device=s.device)).amax(2)
    e = torch.exp(s - m)
    alpha = e / (e @ same)
    intra = torch.einsum('th,hc,hd->tcd', alpha, onehot, g[0])
    f = torch.relu(intra @ W.T + bias) + intra
    lq = scale * torch.einsum('tcd,td->tc', f, qk2)
    beta = torch.softmax(torch.where(cmask[0][None] > 0, lq, torch.tensor(-1e9, dtype=lq.dtype, device=lq.device)), 1)
    return alpha, beta, beta * torch.einsum('tcd,td->tc', f, cand)


def _guarded(shape, dev, pad=1024):
    """a NaN-filled tensor of ``shape`` at the start of a NaN-filled buffer ``pad`` floats longer: (tensor, buffer)"""
    n = int(np.prod(shape))
    buf = torch.full((n + pad,), float('nan'), device=dev)
    return buf[:n].view(*shape), buf


@pytest.mark.parametrize('counts, Hh, C1, D, Au', [
    ([37, 0, 1, 300, 129, 37], 50, 19, 900, 225),      # the default model: empty, single, MIND-sized and long lists
    ([5, 64, 65, 0], 256, 72, 900, 225),               # the limits (the 2-warp CTA); one and two 64-candidate slices
    ([20, 3, 77], 20, 19, 356, 200),                   # hidden_dim 64: D = 356, D % 8 == 4
])
def test_explain_kernel_matches_float64_reference(cuda, counts, Hh, C1, D, Au):
    from nnr_b200 import ops
    Kp, g, W, idx, cmask, Qp, qk2, cand, bias, row_off = _packed_inputs(counts, Hh, C1, D, Au, cuda, seed=sum(counts) + Hh)
    f = lambda x: x.float().contiguous()
    B, n_max, scale = len(counts), max(counts), 1.0 / math.sqrt(Au)
    lds = n_max + 3
    args = (f(Kp), f(g), f(g @ W.T), idx, cmask.to(torch.uint8), row_off, f(Qp), f(qk2), f(cand), f(bias), B, Hh, Au, D,
            C1, n_max, scale)
    scores, s_buf = _guarded((B, lds), cuda)
    alpha, a_buf = _guarded((B, lds, Hh), cuda)
    beta, b_buf = _guarded((B, lds, C1), cuda)
    contrib, c_buf = _guarded((B, lds, C1), cuda)
    ops.cluster_tail_explain_packed(*args, scores, alpha, beta, contrib)
    plain = torch.full((B, lds), float('nan'), device=cuda)
    ops.cluster_tail_scores_packed(*args, plain)
    torch.cuda.synchronize()
    assert torch.equal(_bits(scores), _bits(plain))                                    # the same bits, NaN past the counts
    for buf, t in ((s_buf, scores), (a_buf, alpha), (b_buf, beta), (c_buf, contrib)):
        assert torch.isnan(buf[t.numel():]).all()                                      # nothing written past the tensor
    for b, c in enumerate(counts):
        for t in (alpha, beta, contrib):
            assert torch.isnan(t[b, c:]).all(), b                                      # nor past the count
        if c == 0:
            continue
        r = slice(int(row_off[b]), int(row_off[b + 1]))
        ra, rb, rc = _reference(Kp[b:b + 1], g[b:b + 1], W, idx[b:b + 1], cmask[b:b + 1], Qp[r], qk2[r], cand[r], bias,
                                scale)
        for name, got, ref in (('alpha', alpha[b, :c], ra), ('beta', beta[b, :c], rb), ('contrib', contrib[b, :c], rc)):
            assert rel_err(got, ref) <= 1e-5, (b, name, rel_err(got, ref))
        assert (beta[b, :c][:, cmask[b] == 0] == 0).all()                              # masked clusters: exactly 0


# ---- explain() against the oracle --------------------------------------------------------------------------------------
def _oracle_explain(p, cfg, syn, hist, hl, cand_ids, flags=None):
    """explain_ref.sue_explain on the oracle's own cache, encoded in the same [1, CHUNK] chunks: (alpha, beta,
    beta * f.cand, scores)"""
    from oracle import graph as OG
    t = torch.from_numpy
    with torch.no_grad():
        chunks = []
        for a in range(0, NEWS, CHUNK):
            b = min(NEWS, a + CHUNK)
            chunks.append(O.cne_forward(p, cfg, t(syn.news_title_text[a:b])[None], t(syn.news_title_mask[a:b].copy())[None],
                                        t(syn.news_abstract_text[a:b])[None], t(syn.news_abstract_mask[a:b].copy())[None],
                                        t(syn.news_category[a:b])[None], t(syn.news_subCategory[a:b])[None],
                                        sort_fn=O.stable_sort)[0])
        ocache = torch.cat(chunks)
        g, cm, ci = zip(*[OG.build_history_graph(syn.news_category[hist[b, :hl[b]]], H, cfg.category_num, **(flags or {}))
                          for b in range(len(hl))])
        cand = ocache[t(np.asarray(cand_ids))]
        alpha, beta, fc, user = sue_explain(p, cfg, ocache[t(hist)], t(np.stack(g)), t(np.stack(cm)), t(np.stack(ci)), cand)
        return alpha, beta, None if beta is None else beta * fc, (user * cand).sum(2)


def _check_against_oracle(sc, p, cfg, syn, hist, hl, cand, flags=None):
    ref = _oracle_explain(p, cfg, syn, hist, hl, cand, flags)
    got = {}
    for exact in (True, False):
        e = got[exact] = sc.explain(hist, hl, cand, exact=exact)
        assert torch.equal(_bits(e.scores), _bits(sc.score(hist, hl, cand, exact=exact))), exact
        assert rel_err(e.scores.cpu(), ref[3]) < TOL
        assert rel_err(e.history_weight.cpu(), ref[0]) < TOL, exact
        if ref[1] is None:                                                             # SUE_wo_HCA
            assert e.cluster_weight is None and e.cluster_score is None and e.history_cluster is None
            continue
        assert rel_err(e.cluster_weight.cpu(), ref[1]) < TOL, exact
        assert rel_err(e.cluster_score.cpu(), ref[2]) < TOL, exact
        total = e.cluster_score.sum(2)
        assert ((total - e.scores).abs() <= 1e-6 * e.cluster_score.abs().sum(2)).all(), exact
        _, cmask, cidx = sc._history_graph(torch.as_tensor(hist).to(sc.dev).long(),
                                           torch.as_tensor(hl).to(sc.dev).to(torch.int32))
        cmask[:, -1] = True
        assert torch.equal(e.history_cluster, cidx)
        assert (e.cluster_weight.masked_select(~cmask[:, None, :].expand_as(e.cluster_weight)) == 0).all(), exact
    for name in ('cluster_weight', 'history_weight'):                                  # the two paths agree
        if getattr(got[True], name) is not None:
            assert rel_err(getattr(got[False], name), getattr(got[True], name)) <= 1e-4, name
    return got


@pytest.mark.parametrize('user_encoder', ['SUE', 'SUE_wo_GCN', 'SUE_wo_HCA'])
def test_explain_matches_oracle(cuda, user_encoder):
    cfg = _config(user_encoder=user_encoder)
    p = O.formula_params(cfg)
    syn = _corpus()
    sc = _scorer(_build(cfg, p, cuda), syn)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=4)
    cand = np.random.default_rng(9).integers(0, NEWS, (6, 40))
    _check_against_oracle(sc, p, cfg, syn, hist, hl, cand)


def test_explain_with_a_graph_flag_matches_oracle(sue):
    from nnr_b200 import ops
    from tests.test_pins import FLAG_SETS
    _, syn, p, cfg = sue
    m = sue[0].model
    flags = FLAG_SETS[1]                                                               # asymmetric normalisation
    sc = _scorer(m, syn, graph_flags=ops.graph_flags(**flags))
    hist, hl, _ = syn.sample_behaviors(5, news_num=1, seed=8)
    _check_against_oracle(sc, p, cfg, syn, hist, hl, np.random.default_rng(3).integers(0, NEWS, (5, 30)), flags)


# ---- ragged lists ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('exact', [False, True])
def test_explain_ragged_lists(sue, exact):
    sc, syn, _, _ = sue
    hist, hl, cand, cnt, _, valid = _ragged(syn, 40, 37, seed=5)                       # padding ids -1
    e = sc.explain(hist, hl, cand, cnt, exact=exact)
    v = torch.from_numpy(valid).to(sc.dev)
    for name in ('scores', 'cluster_weight', 'cluster_score', 'history_weight'):
        t = getattr(e, name)
        assert (t[~v] == 0).all(), name                                                # past the counts: 0
    full = sc.explain(hist, hl, np.where(valid, cand, 0), exact=exact)                 # the same entries, nothing padded
    assert rel_err(e.scores[v], full.scores[v]) <= 1e-6
    wide = np.full((40, 60), -1)
    wide[:, :37] = cand
    w = sc.explain(hist, hl, wide, cnt, exact=exact)
    for name in ('scores', 'cluster_weight', 'cluster_score', 'history_weight'):
        a, b = getattr(e, name), getattr(w, name)[:, :37]
        assert rel_err(b[v], a[v]) <= 1e-6, name
        assert (getattr(w, name)[:, 37:] == 0).all(), name
    assert torch.equal(w.history_cluster, e.history_cluster)


# ---- determinism and graph replay --------------------------------------------------------------------------------------
@pytest.mark.parametrize('exact', [False, True])
def test_explain_is_deterministic_and_graph_replay_equals_host_launch(sue, exact):
    sc, syn, _, _ = sue
    hist, hl, cand, cnt, _, _ = _ragged(syn, 70, 24, seed=17)
    a = sc.explain(hist, hl, cand, cnt, exact=exact)
    assert ('explain', exact, (70, hist.shape[1]), (70, 24), sc.cache.data_ptr()) in sc._graphs
    b = sc.explain(hist, hl, cand, cnt, exact=exact)
    c = sc.explain(hist, hl, cand, cnt, exact=exact, cuda_graph=False)
    for name in ('scores', 'cluster_weight', 'cluster_score', 'history_weight'):
        assert torch.equal(_bits(getattr(a, name)), _bits(getattr(b, name))), name
        assert torch.equal(_bits(getattr(a, name)), _bits(getattr(c, name))), name
    assert torch.equal(a.history_cluster, c.history_cluster)


# ---- a recommend() result ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('exact', [False, True])
def test_explain_a_recommend_result(sue, exact):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(64, news_num=1, seed=23)
    hl[0] = H
    others = np.random.default_rng(2).permutation(np.setdiff1d(np.arange(NEWS), hist[0]))[:6]
    pool = np.concatenate([np.unique(hist[0]), others])                                 # user 0: 6 eligible of k = 10
    ids, scores = sc.recommend(hist, hl, pool, 10, exact=exact)
    cnt = (ids >= 0).sum(1)
    assert int(cnt.min()) < 10                                                         # fill entries at some tail
    e = sc.explain(hist, hl, ids, candidate_count=cnt, exact=exact)
    filled = ids >= 0
    assert rel_err(e.scores[filled], scores[filled]) <= 1e-4
    for name in ('scores', 'cluster_weight', 'cluster_score', 'history_weight'):
        assert (getattr(e, name)[~filled] == 0).all(), name
