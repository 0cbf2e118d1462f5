"""GPU tests of the per-category cap of top-k recommendation (CorpusScorer.recommend(max_per_category=m),
nnr_topk_merge_capped).

  * recommend's capped ids and scores equal a numpy reference of the greedy rule applied to score() on the same tiles;
  * m >= k equals the uncapped call bit for bit, through the scorer and kernel against kernel;
  * nnr_topk_merge_capped alone against the reference over several merges: random, tied and +-inf/NaN scores, 1, 18 and
    1024 skewed groups, T = 4096 with k = 1024;
  * after every merge of an adversarial tile sequence (later tiles bring better entries of a group that fills its cap)
    the state equals the reference over the tiles so far;
  * a captured-graph replay of the capped merge equals host launches.
"""
import numpy as np
import pytest
import torch

from tests.test_recommend_gpu import NEWS, _scores, sue, tiled_scores  # noqa: F401  (sue: fixture)

pytestmark = pytest.mark.gpu


def capped_reference(S, groups, eligible, k, m):
    """the greedy rule on a full score matrix S [B, P] (numpy fp32): each row's eligible entries by score descending, ties
    by ascending position, NaN below every number; an entry is taken unless m entries of its group groups[j] were taken
    before it; the first k taken, then (-inf, -1) fill.  Returns (scores [B, k], positions [B, k], groups [B, k])."""
    B, P = S.shape
    out_s = np.full((B, k), -np.inf, dtype=np.float32)
    out_p = np.full((B, k), -1, dtype=np.int64)
    out_g = np.full((B, k), -1, dtype=np.int32)
    for b in range(B):
        pos = np.nonzero(eligible[b])[0]
        v = S[b, pos].astype(np.float64)
        nan = np.isnan(v)
        order = pos[np.lexsort((pos, -np.where(nan, 0.0, v), nan))]
        g = groups[order]
        by_group = np.argsort(g, kind='stable')                  # within a group, still in ranking order
        sg = g[by_group]
        starts = np.r_[0, np.flatnonzero(sg[1:] != sg[:-1]) + 1] if len(sg) else np.zeros(0, dtype=np.int64)
        first = np.repeat(starts, np.diff(np.r_[starts, len(sg)]))
        rank = np.empty(len(g), dtype=np.int64)
        rank[by_group] = np.arange(len(g)) - first               # entries of the same group ranked before this one
        take = order[rank < m][:k]
        out_s[b, :len(take)] = S[b, take]
        out_p[b, :len(take)] = take
        out_g[b, :len(take)] = groups[take]
    return out_s, out_p, out_g


def _eligible(pool, hist, hl, exclude):
    pool = np.asarray(pool)
    hist = np.asarray(hist)
    return np.stack([~np.isin(pool, hist[b, :int(hl[b])]) if exclude else np.ones(len(pool), dtype=bool)
                     for b in range(len(hl))])


def _check_scorer(sc, syn, hist, hl, pool, k, m, T, exclude=True):
    """recommend(max_per_category=m) against the reference on score() of the same tiles: ids and scores exactly equal"""
    ids, scores = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T, max_per_category=m)
    assert ids.shape == (len(hl), k) and ids.dtype == torch.int64 and scores.dtype == torch.float32
    S = tiled_scores(sc, hist, hl, pool, T).cpu().numpy()
    pool = np.asarray(pool)
    rs, rp, rg = capped_reference(S, syn.news_category[pool], _eligible(pool, hist, hl, exclude), k, m)
    rid = np.where(rp >= 0, pool[np.maximum(rp, 0)], -1)
    assert np.array_equal(ids.cpu().numpy(), rid), (ids.cpu().numpy(), rid)
    assert np.array_equal(scores.cpu().numpy(), rs), (scores.cpu().numpy(), rs)
    got = ids.cpu().numpy()
    for b in range(len(hl)):                                      # the cap holds on the result
        real = got[b][got[b] >= 0]
        assert np.bincount(syn.news_category[real]).max(initial=0) <= m
    return got, scores.cpu().numpy()


@pytest.mark.parametrize('B, P, T, k, m, exclude', [
    (6, 150, 64, 10, 1, True),      # P not a multiple of T: two graphed tiles and an eager one
    (6, 150, 64, 10, 2, True),
    (6, 30, 64, 5, 1, True),        # P < T: one partial tile
    (6, 150, 64, 2, 1, True),       # k = 2, m = 1
    (6, 150, 32, 1024, 3, True),    # k at the limit: fill after at most 3 news per category
    (5, 150, 48, 40, 2, False),     # without exclusion
    (70, 100, 32, 12, 2, True),     # score() replays captured graphs too at B >= 64
])
def test_capped_recommend_equals_greedy_reference(sue, B, P, T, k, m, exclude):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=B + P + k)
    pool = np.random.default_rng(P + m).permutation(NEWS)[:P]
    ids, scores = _check_scorer(sc, syn, hist, hl, pool, k, m, T, exclude)
    if k == 1024:
        assert (ids[:, -1] == -1).all() and (scores[:, -1] == -np.inf).all()


def test_capped_recommend_with_duplicate_pool_ids(sue):
    """duplicates are separate entries and each one counts toward its category's cap"""
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(4, news_num=1, seed=5)
    base = np.random.default_rng(1).permutation(NEWS)[:40]
    pool = np.concatenate([base, base[::-1], base[:7]])
    ids, _ = _check_scorer(sc, syn, hist, hl, pool, 30, 2, 32, exclude=False)
    # m = 2: a news duplicated in the pool can fill its category's cap by itself
    assert any(len(set(r[r >= 0].tolist())) < (r >= 0).sum() for r in ids)


def test_capped_recommend_deep_into_a_dominant_category(sue):
    """most of the pool is one category: the cap passes over most of the top of the uncapped order"""
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(5, news_num=1, seed=17)
    cats = syn.news_category
    big = int(np.bincount(cats).argmax())
    own = np.flatnonzero(cats == big)
    rng = np.random.default_rng(6)
    pool = np.concatenate([rng.choice(own, 200), rng.choice(np.flatnonzero(cats != big), 25)])
    pool = rng.permutation(pool)
    assert (cats[pool] == big).mean() > 0.85
    for k, m in ((10, 1), (20, 3)):
        _check_scorer(sc, syn, hist, hl, pool, k, m, 64, exclude=False)
    uncapped, _ = sc.recommend(hist, hl, pool, 20, exclude_history=False, pool_tile=64)
    assert ((cats[uncapped.cpu().numpy()] == big).sum(1) > 3).any()          # without the cap the category crowds the list


def test_capped_recommend_fills_when_too_few_entries_survive_the_cap(sue):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(4, news_num=1, seed=19)
    cats = syn.news_category
    three = np.argsort(np.bincount(cats))[-3:]                    # the three largest categories
    pool = np.flatnonzero(np.isin(cats, three))                   # three categories: at most 3 * m entries survive
    ids, scores = _check_scorer(sc, syn, hist, hl, pool, 10, 2, 16, exclude=False)
    assert (ids[:, 6:] == -1).all() and (scores[:, 6:] == -np.inf).all() and (ids[:, :6] >= 0).all()


def test_cap_of_at_least_k_equals_the_uncapped_call(sue):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=23)
    pool = np.random.default_rng(8).permutation(NEWS)[:140]
    for k in (1, 10, 200):
        ref = sc.recommend(hist, hl, pool, k, pool_tile=32)
        for m in (k, k + 1, 1000):
            got = sc.recommend(hist, hl, pool, k, pool_tile=32, max_per_category=m)
            assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), (k, m)


# ---- the kernel alone ---------------------------------------------------------------------------------------------
NID = 4000


def _inputs(kind, B, P, G, cuda, seed):
    gen = torch.Generator().manual_seed(seed)
    S = _scores(kind, B, P, cuda, gen)
    tile_ids = torch.randint(0, NID, (P,), generator=gen)
    u = torch.rand(NID, generator=gen)
    id_group = (G * u ** 3).long().clamp(max=G - 1).to(torch.int32)     # skewed: low groups hold most news
    pick = torch.randint(0, P, (B, 12), generator=gen)
    excl = tile_ids[pick]                                                # ids that do occur in the pool
    excl_len = torch.randint(0, 13, (B,), generator=gen).to(torch.int32)
    return S, tile_ids.to(cuda), id_group.to(cuda), excl.to(cuda), excl_len.to(cuda)


def _merge_capped(S, tile_ids, excl, excl_len, id_group, G, m, k, T, stop=None):
    from nnr_b200 import ops
    B, P = S.shape
    best_s = torch.empty(B, k, device=S.device)
    best_p = torch.empty(B, k, dtype=torch.int64, device=S.device)
    best_g = torch.empty(B, k, dtype=torch.int32, device=S.device)
    for a in range(0, P if stop is None else stop, T):
        ops.topk_merge_capped(S[:, a:a + T], a, tile_ids[a:a + T], excl, excl_len, id_group, G, m, a == 0, best_s, best_p,
                              best_g)
    return best_s, best_p, best_g


def _kernel_reference(S, tile_ids, excl, excl_len, id_group, m, k):
    S_, ids = S.cpu().numpy(), tile_ids.cpu().numpy()
    if excl is None:
        eligible = np.ones(S_.shape, dtype=bool)
    else:
        x, xl = excl.cpu().numpy(), excl_len.cpu().numpy()
        eligible = np.stack([~np.isin(ids, x[b, :xl[b]]) for b in range(S_.shape[0])])
    return capped_reference(S_, id_group.cpu().numpy()[ids], eligible, k, m)


def _assert_state(got, ref):
    got_s, got_p, got_g = got
    ref_s, ref_p, ref_g = ref
    assert np.array_equal(got_p.cpu().numpy(), ref_p)
    torch.testing.assert_close(got_s.cpu(), torch.from_numpy(ref_s), rtol=0, atol=0, equal_nan=True)
    assert np.array_equal(got_g.cpu().numpy(), ref_g)


@pytest.mark.parametrize('kind', ['random', 'tied', 'inf_nan'])
@pytest.mark.parametrize('B, P, T, k, G, m', [
    (300, 700, 256, 10, 18, 1),        # several merges, a partial last tile
    (300, 700, 256, 10, 18, 2),
    (64, 3 * 4096, 4096, 1024, 1024, 7),   # T and k at their limits, 1024 groups
    (64, 3 * 4096, 4096, 1024, 18, 7),     # at most 18 * 7 entries survive: fill
    (200, 50, 50, 100, 1, 2),          # one group
    (5, 9000, 1000, 1, 18, 1),
    (100, 2000, 500, 64, 1024, 1),
])
def test_capped_merge_matches_reference(cuda, kind, B, P, T, k, G, m):
    S, tile_ids, id_group, excl, excl_len = _inputs(kind, B, P, G, cuda, B + P + k + G + m)
    _assert_state(_merge_capped(S, tile_ids, excl, excl_len, id_group, G, m, k, T),
                  _kernel_reference(S, tile_ids, excl, excl_len, id_group, m, k))
    _assert_state(_merge_capped(S, tile_ids, None, None, id_group, G, m, k, T),
                  _kernel_reference(S, tile_ids, None, None, id_group, m, k))


@pytest.mark.parametrize('kind', ['random', 'tied', 'inf_nan'])
@pytest.mark.parametrize('B, P, T, k', [(300, 700, 256, 10), (64, 3 * 4096, 4096, 1024), (200, 50, 50, 100)])
def test_capped_merge_with_cap_k_equals_uncapped_merge(cuda, kind, B, P, T, k):
    """cap >= k keeps every entry the uncapped merge keeps: the capped kernel's sort and compaction alone"""
    from tests.test_recommend_gpu import _merge_all
    S, tile_ids, id_group, excl, excl_len = _inputs(kind, B, P, 18, cuda, B + P)
    ref_s, ref_p = _merge_all(S, tile_ids, excl, excl_len, k, T)
    for m in (k, k + 3):
        got_s, got_p, got_g = _merge_capped(S, tile_ids, excl, excl_len, id_group, 18, m, k, T)
        assert torch.equal(got_p, ref_p)
        assert torch.equal(got_s.view(torch.int32), ref_s.view(torch.int32))           # bit for bit, NaN included
        want_g = torch.where(ref_p >= 0, id_group[tile_ids[ref_p.clamp(min=0)].long()], torch.full_like(got_g, -1))
        assert torch.equal(got_g, want_g)


def test_capped_merge_adversarial_tiles(cuda):
    """group 0 fills its cap in the state from the first tile; every later tile brings group-0 entries that beat the
    state's, so the earlier ones are evicted and the entries below them move up; groups 1 and 2 get better entries late
    too.  After every merge the state is the reference over the tiles merged so far."""
    B, T, k, m, G, tiles = 8, 64, 12, 2, 6, 8
    gen = torch.Generator().manual_seed(3)
    P = T * tiles
    S = torch.full((B, P), -50.0)
    grp_of_pos = torch.empty(P, dtype=torch.int32)
    for t in range(tiles):
        a = a0 = t * T
        # group 0: 8 entries per tile, each tile's better than the last
        S[:, a:a + 8] = 10.0 * (t + 1) + torch.rand(B, 8, generator=gen)
        grp_of_pos[a:a + 8] = 0
        a += 8
        # groups 1 and 2: better entries in the late tiles, tied within the tile (position order decides)
        for g in (1, 2):
            S[:, a:a + 4] = (5.0 + 3.0 * t * (g == 1) + 2.0 * (t >= tiles - 2)) if t in (0, 3, tiles - 2, tiles - 1) else -60.0
            grp_of_pos[a:a + 4] = g
            a += 4
        # groups 3..5: mid scores from the first tile only, then below every state entry
        S[:, a:a0 + T] = (torch.rand(B, a0 + T - a, generator=gen) * 4 - (0 if t == 0 else 80))
        grp_of_pos[a:a0 + T] = 3 + torch.arange(a0 + T - a, dtype=torch.int32) % 3
    S = S.to(cuda)
    tile_ids = torch.arange(P, device=cuda)                      # news id = pool position: its group is grp_of_pos
    id_group = grp_of_pos.to(cuda)
    evicted = 0
    prev = None
    for stop in range(T, P + 1, T):
        got = _merge_capped(S, tile_ids, None, None, id_group, G, m, k, T, stop=stop)
        _assert_state(got, _kernel_reference(S[:, :stop], tile_ids[:stop], None, None, id_group, m, k))
        pos = set(got[1].flatten().tolist())
        if prev is not None:
            evicted += len(prev - pos)
        prev = pos
        g0 = got[2] == 0
        assert (g0.sum(1) == m).all()                            # group 0 always at its cap, with the newest tile's entries
        assert ((got[1] >= stop - T) | ~g0).all()
    assert evicted >= (tiles - 1) * m


def test_capped_merge_replayed_in_a_graph_equals_host_launch(cuda):
    from nnr_b200 import ops
    B, T, k, G, m = 300, 512, 64, 18, 2
    S, ids, id_group, excl, excl_len = _inputs('tied', B, 2 * T, G, cuda, 0)
    host = _merge_capped(S, ids, excl, excl_len, id_group, G, m, k, T)
    best_s = torch.empty(B, k, device=cuda)
    best_p = torch.empty(B, k, dtype=torch.int64, device=cuda)
    best_g = torch.empty(B, k, dtype=torch.int32, device=cuda)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ops.topk_merge_capped(S[:, :T], 0, ids[:T], excl, excl_len, id_group, G, m, True, best_s, best_p, best_g)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.topk_merge_capped(S[:, :T], 0, ids[:T], excl, excl_len, id_group, G, m, True, best_s, best_p, best_g)
        ops.topk_merge_capped(S[:, T:], T, ids[T:], excl, excl_len, id_group, G, m, False, best_s, best_p, best_g)
    for _ in range(2):
        best_s.fill_(0)
        best_g.fill_(7)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(best_p, host[1]) and torch.equal(best_s, host[0]) and torch.equal(best_g, host[2])
