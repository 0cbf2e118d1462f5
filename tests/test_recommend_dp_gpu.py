"""GPU tests of data-parallel top-k recommendation (CorpusScorer.recommend(collective=True), nnr_topk_merge_lists[_capped]).

  * shards simulated on one GPU: for W = 2, 3, 4, 8 the W rank lists (``_recommend_tiles`` over each rank's contiguous
    share of the tiles) folded by ``_merge_rank_lists`` equal the plain recommend() bit for bit, ids and scores, capped and
    uncapped, for SUE, SUE_wo_HCA and SUE_wo_GCN;
  * nnr_topk_merge_lists[_capped] alone against the numpy reference of the stated order: random, tied and +-inf/NaN
    scores, fill slots inside the lists, real -inf entries, W * k up to 8 * 1024, 1, 18 and 1024 groups; a graph replay
    equals host launches;
  * over NCCL: a group of one rank equals the plain scorer; W = 2 and 4 equal one GPU on every rank; a rank called with a
    different k or pool makes every rank raise, and the next call on the same group succeeds.
"""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_recommend_capped_gpu import capped_reference
from tests.test_recommend_gpu import NEWS, _build, _config, _corpus, _scorer, _scores, sue  # noqa: F401  (sue: fixture)
from tests.test_scoring_dp_gloo import _free_port

pytestmark = pytest.mark.gpu


def _same(a, b):
    """ids equal and scores equal bit for bit (NaN included)"""
    return torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))


def simulated_collective(sc, hist, hl, pool, k, T, W, exclude=True, m=None):
    """recommend(collective=True) over W ranks, on one device: every rank's list, then the final merge"""
    from nnr_b200.scoring import contiguous_blocks
    hid, hl_, pool_, k, T, m_, groups = sc._recommend_inputs(hist, hl, pool, k, exclude, T, m)
    parts = contiguous_blocks(-(-pool_.numel() // T), W)[1]
    lists = [sc._recommend_tiles(hid, hl_, pool_, k, T, a, b, exclude, m_, groups, True) for a, b in parts]
    S, P = torch.stack([x[0] for x in lists]), torch.stack([x[1] for x in lists])
    G = torch.stack([x[2] for x in lists]) if m_ is not None else None
    for (a, b), x in zip(parts, lists):
        if a == b:                                                # a rank without tiles holds the fill list
            assert (x[0] == float('-inf')).all() and (x[1] == -1).all()
    best_s, best_p = sc._merge_rank_lists(S, P, G, m_, groups)
    return sc._pool_ids(pool_, best_p), best_s


def _check(sc, hist, hl, pool, k, T, exclude=True, m=None, worlds=(2, 3, 4, 8)):
    want = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T, max_per_category=m)
    for W in worlds:
        got = simulated_collective(sc, hist, hl, pool, k, T, W, exclude, m)
        assert _same(got, want), (W, got, want)
    return want


@pytest.mark.parametrize('B, P, T, k, exclude', [
    (6, 150, 64, 10, True),         # P not a multiple of T: 3 tiles, ranks without tiles at W = 4 and 8
    (6, 150, 16, 10, True),         # 10 tiles: several per rank
    (6, 30, 64, 5, True),           # one tile, fewer tiles than ranks
    (6, 150, 16, 1, True),          # k = 1
    (6, 150, 32, 1024, True),       # k at the limit: fill
    (1, 150, 16, 20, True),         # one user
    (5, 150, 48, 40, False),        # without exclusion
])
@pytest.mark.parametrize('m', [None, 1, 2])
def test_simulated_ranks_equal_plain_recommend(sue, B, P, T, k, exclude, m):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=B + P + k)
    pool = np.random.default_rng(P + T).permutation(NEWS)[:P]
    ids, scores = _check(sc, hist, hl, pool, k, T, exclude, m)
    if k == 1024:
        assert (ids[:, -1] == -1).all() and (scores[:, -1] == float('-inf')).all()


@pytest.mark.parametrize('m', [None, 2])
def test_simulated_ranks_with_duplicate_pool_ids(sue, m):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(4, news_num=1, seed=5)
    base = np.random.default_rng(1).permutation(NEWS)[:40]
    pool = np.concatenate([base, base[::-1], base[:7]])        # duplicates land in different ranks' tiles
    ids, _ = _check(sc, hist, hl, pool, 30, 16, exclude=False, m=m)
    assert any(len(set(r[r >= 0].tolist())) < (r >= 0).sum() for r in ids.cpu().numpy())


@pytest.mark.parametrize('m', [1, 2])
def test_simulated_ranks_with_a_dominant_category(sue, m):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(5, news_num=1, seed=17)
    cats = syn.news_category
    big = int(np.bincount(cats).argmax())
    rng = np.random.default_rng(6)
    pool = rng.permutation(np.concatenate([rng.choice(np.flatnonzero(cats == big), 200),
                                           rng.choice(np.flatnonzero(cats != big), 25)]))
    ids, _ = _check(sc, hist, hl, pool, 20, 32, exclude=False, m=m)
    got = ids.cpu().numpy()
    assert all(np.bincount(cats[r[r >= 0]]).max(initial=0) <= m for r in got)


@pytest.mark.parametrize('user_encoder', ['SUE_wo_HCA', 'SUE_wo_GCN'])
def test_simulated_ranks_other_user_encoders(cuda, user_encoder):
    from oracle import nnr_oracle as O
    cfg = _config(user_encoder=user_encoder)
    syn = _corpus()
    sc = _scorer(_build(cfg, O.formula_params(cfg), cuda), syn)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=4)
    pool = np.random.default_rng(9).permutation(NEWS)[:130]
    for m in (None, 2):
        _check(sc, hist, hl, pool, 12, 32, m=m)


# ---- the list merge alone ------------------------------------------------------------------------------------------
def _rank_lists(S, groups, eligible, k, m, W, seed, shuffle):
    """W reference best lists of a random partition of the positions [0, P) (numpy): scores, global positions and groups
    [W, B, k], fill slots (-inf, -1, -1) where fewer than k entries are eligible; shuffle: entries and fill slots in random
    order within each list row"""
    B, P = S.shape
    rng = np.random.default_rng(seed)
    owner = rng.integers(0, W, P)
    out = [np.zeros((W, B, k), dtype=t) for t in (np.float32, np.int64, np.int32)]
    for r in range(W):
        cols = np.flatnonzero(owner == r)
        s, p, g = capped_reference(S[:, cols], groups[cols], eligible[:, cols], k, m)
        p = np.where(p >= 0, cols[np.maximum(p, 0)], -1)
        if shuffle:
            perm = np.argsort(rng.random((B, k)), 1)
            s, p, g = (np.take_along_axis(x, perm, 1) for x in (s, p, g))
        out[0][r], out[1][r], out[2][r] = s, p, g
    return out


def _merge_lists(S, P, G, num_groups, m, dev):
    from nnr_b200 import ops
    W, B, k = S.shape
    S, P = torch.from_numpy(S).to(dev), torch.from_numpy(P).to(dev)
    best_s = torch.empty(B, k, device=dev)
    best_p = torch.empty(B, k, dtype=torch.int64, device=dev)
    best_g = torch.empty(B, k, dtype=torch.int32, device=dev)
    for r in range(W):
        if m is None:
            ops.topk_merge_lists(S[r], P[r], r == 0, best_s, best_p)
        else:
            ops.topk_merge_lists_capped(S[r], P[r], torch.from_numpy(G[r]).to(dev), num_groups, m, r == 0, best_s, best_p,
                                        best_g)
    return best_s, best_p, best_g


@pytest.mark.parametrize('kind', ['random', 'tied', 'inf_nan'])
@pytest.mark.parametrize('B, P, W, k, G, m, shuffle', [
    (300, 700, 4, 10, 18, None, False),
    (300, 700, 3, 10, 18, 1, True),            # fill and entries in random order within each list
    (300, 700, 2, 10, 18, 2, False),
    (16, 8 * 1300, 8, 1024, 1024, None, False),  # W * k = 8 * 1024
    (16, 8 * 1300, 8, 1024, 1024, 3, True),
    (16, 8 * 1300, 8, 1024, 18, 7, False),     # at most 18 * 7 entries survive: fill
    (200, 50, 8, 100, 1, 2, False),            # one group; lists mostly fill
    (5, 9000, 5, 1, 18, 1, False),
])
def test_list_merge_matches_reference(cuda, kind, B, P, W, k, G, m, shuffle):
    gen = torch.Generator().manual_seed(B + P + W + k)
    S = _scores(kind, B, P, 'cpu', gen).numpy()
    rng = np.random.default_rng(B + k)
    groups = (G * rng.random(P) ** 3).astype(np.int32).clip(max=G - 1)
    eligible = rng.random((B, P)) > 0.2
    lists = _rank_lists(S, groups, eligible, k, k if m is None else m, W, B + P, shuffle)
    got_s, got_p, got_g = _merge_lists(*lists, G, m, cuda)
    ref_s, ref_p, ref_g = capped_reference(S, groups, eligible, k, k if m is None else m)
    assert np.array_equal(got_p.cpu().numpy(), ref_p)
    assert np.array_equal(got_s.cpu().numpy().view(np.int32), ref_s.view(np.int32))
    if m is not None:
        assert np.array_equal(got_g.cpu().numpy(), ref_g)


@pytest.mark.parametrize('m', [None, 1])
def test_list_merge_ranks_real_minus_inf_before_the_fill(cuda, m):
    """lists that hold a few numbers, then real -inf entries, then fill: every -inf entry is kept ahead of the fill, in
    position order, and the fill slots count toward nothing"""
    B, k, W = 3, 8, 3
    S = np.full((W, B, k), -np.inf, dtype=np.float32)
    P = np.full((W, B, k), -1, dtype=np.int64)
    G = np.full((W, B, k), -1, dtype=np.int32)
    for r in range(W):
        S[r, :, 0] = 1.0 + r                                  # one number per list
        P[r, :, 0] = 100 + r
        P[r, :, 1:3] = [10 * r + 5, 10 * r + 1]                # two real -inf entries, then fill
        G[r, :, :3] = [0, r + 1, r + 1]
    got_s, got_p, _ = _merge_lists(S, P, G, 4, m, cuda)
    if m is None:
        want_p = [102, 101, 100, 1, 5, 11, 15, 21]
    else:                                                      # one per group: 0 from the best number, then 1, 2, 3
        want_p = [102, 1, 11, 21, -1, -1, -1, -1]
    assert (got_p.cpu().numpy() == want_p).all(), got_p
    n_num = 3 if m is None else 1
    assert (got_s[:, :n_num] > 0).all() and (got_s[:, n_num:] == float('-inf')).all()


def test_list_merge_replayed_in_a_graph_equals_host_launch(cuda):
    from nnr_b200 import ops
    B, P, W, k, G, m = 300, 3000, 4, 64, 18, 2
    gen = torch.Generator().manual_seed(0)
    S = _scores('tied', B, P, 'cpu', gen).numpy()
    groups = np.random.default_rng(0).integers(0, G, P).astype(np.int32)
    lists = _rank_lists(S, groups, np.ones((B, P), dtype=bool), k, m, W, 1, True)
    for mm in (None, m):
        host = _merge_lists(*lists, G, mm, cuda)
        Sd, Pd, Gd = (torch.from_numpy(x).to(cuda) for x in lists)
        best = (torch.empty(B, k, device=cuda), torch.empty(B, k, dtype=torch.int64, device=cuda),
                torch.empty(B, k, dtype=torch.int32, device=cuda))

        def merges():
            for r in range(W):
                if mm is None:
                    ops.topk_merge_lists(Sd[r], Pd[r], r == 0, *best[:2])
                else:
                    ops.topk_merge_lists_capped(Sd[r], Pd[r], Gd[r], G, mm, r == 0, *best)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            merges()
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            merges()
        for _ in range(2):
            best[0].fill_(0)
            best[1].fill_(7)
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(best[1], host[1]) and torch.equal(best[0].view(torch.int32), host[0].view(torch.int32))
            if mm is not None:
                assert torch.equal(best[2], host[2])


# ---- over NCCL -------------------------------------------------------------------------------------------------------
def _worker(rank, world, port, q, case):
    try:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        torch.cuda.set_device(rank)
        dev = torch.device('cuda', rank)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
        from oracle import nnr_oracle as O
        cfg = _config()
        m = _build(cfg, O.formula_params(cfg), dev)
        syn = _corpus()
        ref = _scorer(m, syn)
        sh = _scorer(m, syn, process_group=dist.group.WORLD)
        hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=31)
        if case == 'equal':
            for P, T, k, cap, exclude, graph in [
                (150, 64, 10, None, True, True),       # 3 tiles: a partial one, and a rank without tiles at W = 4
                (150, 16, 10, None, True, True),
                (150, 16, 10, 1, True, True),
                (150, 32, 1024, 2, True, False),       # fill
                (30, 64, 5, None, False, True),        # one tile
                (150, 16, 40, 2, False, True),
                (0, 16, 4, None, True, True),          # empty pool
            ]:
                pool = np.random.default_rng(P + T).permutation(NEWS)[:P]
                want = ref.recommend(hist, hl, pool, k, exclude, T, cuda_graph=graph, max_per_category=cap)
                got = sh.recommend(hist, hl, pool, k, exclude, T, cuda_graph=graph, max_per_category=cap, collective=True)
                assert _same(got, want), (P, T, k, cap, exclude)
            want = ref.recommend(hist[:1], hl[:1], np.arange(NEWS), 20)        # one user, the default tile
            assert _same(sh.recommend(hist[:1], hl[:1], np.arange(NEWS), 20, collective=True), want)
            if rank == 0:                                     # without collective=True: rank-local
                assert _same(sh.recommend(hist, hl, np.arange(NEWS), 7), ref.recommend(hist, hl, np.arange(NEWS), 7))
            dist.barrier()
        else:
            pool = np.arange(100)
            with pytest.raises(RuntimeError, match=r'k: \[10, 11\]'):
                sh.recommend(hist, hl, pool, 10 + rank, pool_tile=16, collective=True)
            other = pool.copy()
            other[5] += rank
            with pytest.raises(RuntimeError, match='pool_ids checksum'):
                sh.recommend(hist, hl, other, 10, pool_tile=16, collective=True)
            with pytest.raises(RuntimeError, match='argument error'):
                sh.recommend(hist, hl, pool, 10, pool_tile=16 if rank == 0 else 0, collective=True)
            got = sh.recommend(hist, hl, pool, 10, pool_tile=16, collective=True)     # the group still works
            assert _same(got, ref.recommend(hist, hl, pool, 10, pool_tile=16))
        torch.cuda.synchronize()
        q.put((rank, 'ok'))
    except BaseException as ex:                               # surface the failure in the parent
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        import sys
        sys.stdout.flush()
        q.close()
        q.join_thread()
        os._exit(0)


def _run(world, case):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip('needs %d GPUs, found %d' % (world, torch.cuda.device_count() if torch.cuda.is_available() else 0))
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, case)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = [q.get(timeout=600) for _ in range(world)]
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    for rank, msg in sorted(results):
        assert msg == 'ok', 'rank %d: %s' % (rank, msg)


def test_collective_group_of_one_rank_equals_plain_recommend():
    _run(1, 'equal')


@pytest.mark.parametrize('world', [2, 4])
def test_collective_recommend_equals_one_gpu(world):
    _run(world, 'equal')


def test_ranks_called_with_different_arguments_all_raise():
    _run(2, 'mismatch')
