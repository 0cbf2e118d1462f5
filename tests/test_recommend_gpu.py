"""GPU tests of top-k news recommendation over a candidate pool (CorpusScorer.recommend, nnr_topk_merge).

  * recommend's scores are bit-identical to score() on the same tiles, and its ids / scores equal a stable descending sort
    of the concatenated score() rows with the exclusions applied;
  * the scores match the fp64-grade oracle (oracle.sue_forward on the same corpus chunks) for SUE, SUE_wo_HCA, SUE_wo_GCN
    and for graphs built with every non-default graph flag set;
  * nnr_topk_merge alone against a torch reference of the stated order;
  * captured-graph replays equal host launches; memory does not grow with the pool.
"""
import numpy as np
import pytest
import torch

from oracle import nnr_oracle as O
from tests.util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-4
NEWS, H, CHUNK = 150, 8, 64


def _build(cfg, params, dev):
    import nnr_b200
    from nnr_b200 import engine
    engine.sort_fn = O.stable_sort                       # same tie-breaking as the oracle
    cfg.pretrained_word_embedding = params['news_encoder.word_embedding.weight']
    m = nnr_b200.Model(cfg)
    m.initialize()
    m.load_state_dict(O.alias_state_dict(params), strict=True)
    m.to(dev).eval()
    return m


def _corpus():
    from nnr_b200.synthetic import SyntheticMIND
    return SyntheticMIND(news_num=NEWS, vocabulary_size=600, subCategory_num=30, max_title_length=10, max_abstract_length=20,
                         max_history_num=H, lengths='uniform', seed=21)


def _config(**kw):
    return O.make_config(vocabulary_size=600, max_history_num=H, max_title_length=10, max_abstract_length=20,
                         subCategory_num=30, gcn_layer_num=2, **kw)


def _scorer(m, syn, **kw):
    from nnr_b200.scoring import CorpusScorer
    sc = CorpusScorer(m, syn.news_title_text, syn.news_title_mask, syn.news_abstract_text, syn.news_abstract_mask,
                      syn.news_category, syn.news_subCategory, chunk=CHUNK, **kw)
    sc.encode_corpus()
    return sc


@pytest.fixture(scope='module')
def sue(cuda):
    cfg = _config()
    p = O.formula_params(cfg)
    syn = _corpus()
    return _scorer(_build(cfg, p, cuda), syn), syn, p, cfg


def stated_order(S, pool, hist, hl, k, exclude):
    """the contract of recommend() on a full score matrix S [B, P]: eligible entries by score descending, ties by
    ascending pool position, NaN below every number, then (-1, -inf) fill.  numpy, row by row."""
    S = S.cpu().numpy()
    pool = np.asarray(pool)
    B, P = S.shape
    ids = np.full((B, k), -1, dtype=np.int64)
    scores = np.full((B, k), -np.inf, dtype=np.float32)
    for b in range(B):
        elig = np.ones(P, dtype=bool)
        if exclude:
            elig &= ~np.isin(pool, np.asarray(hist)[b, :int(hl[b])])
        pos = np.nonzero(elig)[0]
        v = S[b, pos].astype(np.float64)
        nan = np.isnan(v)
        take = pos[np.lexsort((pos, -np.where(nan, 0.0, v), nan))][:k]
        ids[b, :len(take)] = pool[take]
        scores[b, :len(take)] = S[b, take]
    return torch.from_numpy(ids), torch.from_numpy(scores)


def tiled_scores(sc, hist, hl, pool, T):
    """score() of every pool tile, expanded over the users: the same shapes as recommend's tiles"""
    B = len(hl)
    pool = torch.as_tensor(pool)
    return torch.cat([sc.score(hist, hl, pool[a:a + T].expand(B, -1)) for a in range(0, len(pool), T)], 1)


def _check_equal_to_score(sc, hist, hl, pool, k, T, exclude=True):
    ids, scores = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T)
    assert ids.shape == (len(hl), k) and ids.dtype == torch.int64 and scores.dtype == torch.float32
    rid, rscore = stated_order(tiled_scores(sc, hist, hl, pool, T), pool, hist, hl, k, exclude)
    assert torch.equal(ids.cpu(), rid), (ids.cpu(), rid)
    assert torch.equal(scores.cpu(), rscore), (scores.cpu(), rscore)
    return ids.cpu(), scores.cpu()


@pytest.mark.parametrize('B, P, T, k', [
    (6, 150, 64, 10),         # P not a multiple of T: two graphed tiles and an eager one
    (6, 30, 64, 5),           # P < T: one partial tile
    (6, 150, 64, 1),
    (6, 150, 32, 1024),       # k at the limit and above the number of eligible entries: fill
    (1, 150, 16, 20),         # one user
    (70, 100, 32, 12),        # score() replays captured graphs too at B >= 64
])
def test_recommend_is_a_stable_sort_of_tiled_score(sue, B, P, T, k):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=B + P)
    pool = np.random.default_rng(P).permutation(NEWS)[:P]
    ids, scores = _check_equal_to_score(sc, hist, hl, pool, k, T)
    if k > P:
        assert (ids[:, P:] == -1).all() and (scores[:, P:] == float('-inf')).all()


def test_recommend_without_exclusion(sue):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(5, news_num=1, seed=3)
    _check_equal_to_score(sc, hist, hl, np.arange(NEWS), 40, 48, exclude=False)


def test_duplicate_pool_ids_tie_break_by_position(sue):
    """a duplicated id scores exactly the same at both positions: the earlier position ranks first"""
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(4, news_num=1, seed=5)
    base = np.random.default_rng(1).permutation(NEWS)[:40]
    pool = np.concatenate([base, base[::-1], base[:7]])
    ids, _ = _check_equal_to_score(sc, hist, hl, pool, 60, 32, exclude=False)
    assert all(len(set(r.tolist())) < 60 for r in ids)          # the duplicates are returned as separate entries


def test_user_whose_whole_history_is_in_the_pool(sue):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(3, news_num=1, seed=7)
    hl[0] = H
    own = hist[0, :H]
    others = np.setdiff1d(np.arange(NEWS), own)[:20]
    pool = np.concatenate([own, others])
    ids, scores = _check_equal_to_score(sc, hist, hl, pool, len(pool), 16)
    assert not np.isin(ids[0].numpy(), own).any()
    eligible0 = len(others)
    assert (ids[0, eligible0:] == -1).all() and (ids[0, :eligible0] >= 0).all()
    # a pool made only of the user's history leaves nothing eligible
    ids, scores = sc.recommend(hist[:1], hl[:1], own, 4)
    assert (ids == -1).all() and (scores == float('-inf')).all()


def _oracle_scores(p, cfg, syn, hist, hl, pool, flags=None):
    """oracle.sue_forward on the oracle's own cache, encoded in the same [1, CHUNK] chunks"""
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
        B = len(hl)
        g, cm, ci = zip(*[OG.build_history_graph(syn.news_category[hist[b, :hl[b]]], H, cfg.category_num, **(flags or {}))
                          for b in range(B)])
        cand = ocache[t(np.asarray(pool))].unsqueeze(0).expand(B, -1, -1)
        user = O.sue_forward(p, cfg, ocache[t(hist)], t(np.stack(g)), t(np.stack(cm)), t(np.stack(ci)), cand)
        return (user * cand).sum(2)


def _recommend_all(sc, hist, hl, pool, T):
    """every pool entry's score from recommend (k = P, no exclusion), back in pool order (the pool ids are distinct)"""
    ids, scores = sc.recommend(hist, hl, pool, len(pool), exclude_history=False, pool_tile=T)
    where = {int(i): j for j, i in enumerate(pool)}
    out = torch.empty(len(hl), len(pool))
    for b in range(len(hl)):
        out[b, [where[int(i)] for i in ids[b]]] = scores[b].cpu()
    return out


@pytest.mark.parametrize('user_encoder', ['SUE', 'SUE_wo_HCA', 'SUE_wo_GCN'])
def test_recommend_scores_match_oracle(cuda, user_encoder):
    cfg = _config(user_encoder=user_encoder)
    p = O.formula_params(cfg)
    syn = _corpus()
    sc = _scorer(_build(cfg, p, cuda), syn)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=4)
    pool = np.random.default_rng(9).permutation(NEWS)[:70]
    assert rel_err(_recommend_all(sc, hist, hl, pool, 32), _oracle_scores(p, cfg, syn, hist, hl, pool)) < TOL


def test_recommend_with_graph_flags_matches_oracle(sue, cuda):
    from nnr_b200 import ops
    from tests.test_pins import FLAG_SETS
    _, syn, p, cfg = sue
    m = _build(cfg, p, cuda)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=8)
    pool = np.random.default_rng(3).permutation(NEWS)[:50]
    default = None
    for flags in FLAG_SETS:
        sc = _scorer(m, syn, graph_flags=ops.graph_flags(**flags))
        got = _recommend_all(sc, hist, hl, pool, 32)
        assert rel_err(got, _oracle_scores(p, cfg, syn, hist, hl, pool, flags)) < TOL, flags
        if default is None:
            default = got
        else:
            assert not torch.equal(got, default), flags          # the flag reaches the graph


def _reference_topk(S, tile_ids, excl, excl_len, k):
    """torch reference of nnr_topk_merge over the whole row S [B, P]: returns (scores [B, k], positions [B, k])"""
    B, P = S.shape
    h = torch.arange(excl.shape[1], device=S.device)
    excluded = torch.zeros(B, P, dtype=torch.bool, device=S.device)
    for j in range(excl.shape[1]):
        excluded |= (tile_ids[None, :] == excl[:, j:j + 1]) & (h[j] < excl_len[:, None])
    nan = torch.isnan(S)
    v = torch.where(nan | excluded, torch.full_like(S, float('-inf')), S)
    order = torch.sort(v, dim=1, descending=True, stable=True)[1]
    cls = (nan.to(torch.int8) + 2 * excluded.to(torch.int8)).clamp(max=2)      # 0 number, 1 NaN, 2 not eligible
    order = torch.gather(order, 1, torch.sort(torch.gather(cls, 1, order), dim=1, stable=True)[1])[:, :k]
    cls_k = torch.gather(cls, 1, order)
    pos = torch.where(cls_k == 2, torch.full_like(order, -1), order)
    sc = torch.where(cls_k == 2, torch.full_like(S[:, :k], float('-inf')), torch.gather(S, 1, order))
    if k > P:
        pad = k - P
        pos = torch.cat([pos, torch.full((B, pad), -1, dtype=pos.dtype, device=S.device)], 1)
        sc = torch.cat([sc, torch.full((B, pad), float('-inf'), device=S.device)], 1)
    return sc, pos


def _merge_all(S, tile_ids, excl, excl_len, k, T):
    from nnr_b200 import ops
    B, P = S.shape
    best_s = torch.empty(B, k, device=S.device)
    best_p = torch.empty(B, k, dtype=torch.int64, device=S.device)
    for a in range(0, P, T):
        ops.topk_merge(S[:, a:a + T], a, tile_ids[a:a + T], excl, excl_len, a == 0, best_s, best_p)
    return best_s, best_p


def _scores(kind, B, P, dev, gen):
    if kind == 'random':
        return torch.randn(B, P, generator=gen).to(dev)
    if kind == 'tied':
        return (torch.randint(-3, 4, (B, P), generator=gen).float() / 2).to(dev)
    S = torch.randint(-2, 3, (B, P), generator=gen).float()
    r = torch.rand(B, P, generator=gen)
    S[r < 0.2] = float('-inf')
    S[(r >= 0.2) & (r < 0.35)] = float('nan')
    S[(r >= 0.35) & (r < 0.4)] = float('inf')
    S[(r >= 0.4) & (r < 0.45)] = -0.0
    return S.to(dev)


@pytest.mark.parametrize('kind', ['random', 'tied', 'inf_nan'])
@pytest.mark.parametrize('B, P, T, k', [
    (3000, 700, 256, 10),      # thousands of rows, several tiles, a partial last one
    (64, 3 * 4096, 4096, 1024),  # T and k at their limits, three merges
    (200, 50, 50, 100),        # k above P: fill
    (5, 9000, 1000, 1),
])
def test_topk_merge_matches_torch_reference(cuda, kind, B, P, T, k):
    gen = torch.Generator().manual_seed(B + P + k)
    S = _scores(kind, B, P, cuda, gen)
    tile_ids = torch.randint(0, 400, (P,), generator=gen).to(cuda)
    excl = torch.randint(0, 400, (B, 12), generator=gen).to(cuda)
    excl_len = torch.randint(0, 13, (B,), generator=gen).to(torch.int32).to(cuda)
    got_s, got_p = _merge_all(S, tile_ids, excl, excl_len, k, T)
    ref_s, ref_p = _reference_topk(S, tile_ids, excl, excl_len, k)
    assert torch.equal(got_p, ref_p)
    torch.testing.assert_close(got_s, ref_s, rtol=0, atol=0, equal_nan=True)
    # without an exclusion list every entry is eligible
    got_s, got_p = _merge_all(S, tile_ids, None, None, k, T)
    ref_s, ref_p = _reference_topk(S, tile_ids, excl[:, :0], excl_len, k)
    assert torch.equal(got_p, ref_p)
    torch.testing.assert_close(got_s, ref_s, rtol=0, atol=0, equal_nan=True)


def test_topk_merge_replayed_in_a_graph_equals_host_launch(cuda):
    from nnr_b200 import ops
    gen = torch.Generator().manual_seed(0)
    B, T, k = 300, 512, 64
    S = _scores('tied', B, 2 * T, cuda, gen)
    ids = torch.randint(0, 100, (2 * T,), generator=gen).to(cuda)
    excl = torch.randint(0, 100, (B, 10), generator=gen).to(cuda)
    excl_len = torch.full((B,), 10, dtype=torch.int32, device=cuda)
    host_s, host_p = _merge_all(S, ids, excl, excl_len, k, T)
    best_s = torch.empty(B, k, device=cuda)
    best_p = torch.empty(B, k, dtype=torch.int64, device=cuda)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.topk_merge(S[:, :T], 0, ids[:T], excl, excl_len, True, best_s, best_p)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.topk_merge(S[:, :T], 0, ids[:T], excl, excl_len, True, best_s, best_p)
        ops.topk_merge(S[:, T:], T, ids[T:], excl, excl_len, False, best_s, best_p)
    for _ in range(2):
        best_s.fill_(0)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(best_p, host_p) and torch.equal(best_s, host_s)


def test_recommend_graph_replay_equals_host_launched(sue):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(9, news_num=1, seed=11)
    pool = np.random.default_rng(2).permutation(NEWS)[:140]
    eager = sc.recommend(hist, hl, pool, 25, pool_tile=32, cuda_graph=False)
    graphed = sc.recommend(hist, hl, pool, 25, pool_tile=32)
    assert ('recommend', 9, H, 32, sc.cache.data_ptr()) in sc._graphs
    hist2, hl2, _ = syn.sample_behaviors(9, news_num=1, seed=12)
    other = sc.recommend(hist2, hl2, pool, 25, pool_tile=32)            # replays with another user side
    again = sc.recommend(hist, hl, pool, 25, pool_tile=32)
    for a, b in ((eager, graphed), (eager, again)):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(other[1], sc.recommend(hist2, hl2, pool, 25, pool_tile=32, cuda_graph=False)[1])


@pytest.mark.parametrize('cuda_graph', [False, True])
def test_recommend_memory_does_not_grow_with_the_pool(sue, cuda_graph):
    sc, syn, _, _ = sue
    B, T = 32, 64
    hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=13)
    pool = torch.from_numpy(np.random.default_rng(4).integers(0, NEWS, 8 * T))

    def peak(P):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        sc.recommend(hist, hl, pool[:P], 10, pool_tile=T, cuda_graph=cuda_graph)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base
    peak(T), peak(8 * T)                                                 # warm-up: graph capture, workspaces
    one, eight = peak(T), peak(8 * T)
    tail = B * T * 19 * 900 * 4                                         # one D-wide fp32 buffer of the cluster tail
    # host-launched tiles allocate the tail per tile; a captured graph holds it in its own pool, allocated at capture
    assert cuda_graph or one > tail, (one, tail)
    assert eight <= 1.03 * one + 65536, (one, eight)
