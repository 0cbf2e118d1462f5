"""CPU test of the host logic of CorpusScorer.recommend(collective=True) over gloo, world sizes 2, 3 and 4: the tile
partition, the fill list of ranks without tiles, the all-gather layout of the rank lists, the input-agreement check, and
that the group keeps working after a rejected call.  The user encoder is a torch fake whose scores tie often, and the
four top-k merges (nnr_topk_merge[_capped], nnr_topk_merge_lists[_capped]) are replaced by a torch fake of the stated
order, so the collective result must equal the plain scorer's bit for bit.  tests/test_recommend_dp_gpu.py runs the
real kernels, and the real model over NCCL."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_scoring_dp_gloo import _corpus, _Encoder, _free_port


class _UserEncoder(torch.nn.Module):
    category_num = 19                                          # 18 categories: the capped merge's groups

    def user_side(self, hist, graph, cmask, cidx):
        return (hist.sum(1),)

    def tile_scores(self, user, cand):
        s = torch.round((cand * user[0][:, None, :]).sum(2) / 4000.0)    # coarse: many ties within and across tiles
        s[:, ::7] = float('nan')
        s[:, 3::11] = float('-inf')
        return s


class _Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.news_encoder = _Encoder()
        self.user_encoder = _UserEncoder()
        self.w = torch.nn.Parameter(torch.zeros(1))


def _scorer_class():
    from nnr_b200.scoring import CorpusScorer

    class CpuScorer(CorpusScorer):
        def _check_group(self):                               # gloo and CPU tensors: the host logic only
            pass

        def _history_graph(self, hid, hl):
            return None, None, None
    return CpuScorer


def _fold(best_s, best_p, best_g, s, p, g, init, cap):
    """the stated order on the running list plus the new entries s / p / g [B, n] (p < 0: empty): score descending, ties
    by ascending position, NaN last; with a cap, an entry is taken unless cap entries of its group were taken"""
    k = best_s.shape[1]
    for b in range(best_s.shape[0]):
        ent = [] if init else [(float(best_s[b, i]), int(best_p[b, i]), None if best_g is None else int(best_g[b, i]))
                               for i in range(k) if best_p[b, i] >= 0]
        ent += [(float(s[b, j]), int(p[b, j]), None if g is None else int(g[b, j])) for j in range(s.shape[1]) if p[b, j] >= 0]
        ent.sort(key=lambda e: (np.isnan(e[0]), 0.0 if np.isnan(e[0]) else -e[0], e[1]))
        taken, count = [], {}
        for e in ent:
            if cap is None or count.get(e[2], 0) < cap:
                taken.append(e)
                count[e[2]] = count.get(e[2], 0) + 1
            if len(taken) == k:
                break
        best_s[b] = float('-inf')
        best_p[b] = -1
        if best_g is not None:
            best_g[b] = -1
        for i, e in enumerate(taken):
            best_s[b, i], best_p[b, i] = e[0], e[1]
            if best_g is not None:
                best_g[b, i] = e[2]


def _fake_ops(ops, calls):
    """torch fakes of the four merges; the tile merges record their pool offset in ``calls``"""
    def tile(scores, pos0, tile_ids, exclude, exclude_len, init, best_s, best_p, id_group=None, cap=None, best_g=None):
        calls.append(int(pos0))
        B, T = scores.shape
        p = (pos0 + torch.arange(T)).expand(B, T).clone()
        if exclude is not None:
            for b in range(B):
                p[b, torch.isin(tile_ids, exclude[b, :int(exclude_len[b])])] = -1
        g = None if id_group is None else id_group[tile_ids].expand(B, T)
        _fold(best_s, best_p, best_g, scores, p, g, init, cap)

    ops.topk_merge = tile
    ops.topk_merge_capped = lambda s, a, ids, x, xl, idg, G, m, init, bs, bp, bg: tile(s, a, ids, x, xl, init, bs, bp, idg, m, bg)
    ops.topk_merge_lists = lambda s, p, init, bs, bp: _fold(bs, bp, None, s, p, None, init, None)
    ops.topk_merge_lists_capped = lambda s, p, g, G, m, init, bs, bp, bg: _fold(bs, bp, bg, s, p, g, init, m)


def _same(a, b):
    """ids and score bits equal (a NaN equals a NaN of the same bits)"""
    return torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))


def _worker(rank, world, port, q):
    try:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        dist.init_process_group('gloo', rank=rank, world_size=world)
        from nnr_b200 import ops
        from nnr_b200.scoring import contiguous_blocks
        calls = []
        _fake_ops(ops, calls)
        Scorer = _scorer_class()
        m = _Model()
        fields = _corpus(120, seed=120)
        ref, sh = Scorer(m, *fields, chunk=64), Scorer(m, *fields, chunk=64, process_group=dist.group.WORLD)
        ref.encode_corpus(cuda_graph=False)
        sh.encode_corpus(cuda_graph=False)
        rng = np.random.default_rng(4)
        hist = rng.integers(0, 120, size=(5, 6))
        hl = np.array([0, 6, 3, 1, 5])
        dup = np.concatenate([np.arange(0, 40), np.arange(0, 20)])
        for P, T, k, cap, exclude, pool in [
            (50, 8, 5, None, True, None),           # 7 tiles, the last one partial
            (50, 8, 5, 1, True, None),
            (50, 8, 12, 2, False, None),
            (5, 4, 3, None, False, None),           # 2 tiles: ranks without tiles at world 3 and 4
            (5, 4, 3, 1, True, None),
            (30, 30, 40, 2, True, None),            # one tile, k above the eligible entries: fill
            (60, 16, 30, None, False, dup),         # duplicate pool ids
            (60, 16, 1, 1, False, dup),
            (0, 8, 4, None, True, None),            # an empty pool: the fill on every rank
        ]:
            pool = np.random.default_rng(P).permutation(120)[:P] if pool is None else pool
            want = ref.recommend(hist, hl, pool, k, exclude, T, cuda_graph=False, max_per_category=cap)
            del calls[:]
            got = sh.recommend(hist, hl, pool, k, exclude, T, cuda_graph=False, max_per_category=cap, collective=True)
            case = (P, T, k, cap, exclude)
            assert _same(got, want), (case, got, want)
            first, end = contiguous_blocks(-(-P // T), world)[1][rank]
            assert calls == list(range(first * T, min(end * T, P), T)), (case, calls)      # this rank's tiles only
            if P == 0:
                assert got[0].dtype == torch.int64 and (got[0] == -1).all() and (got[1] == float('-inf')).all()
        # a rank without tiles contributes the fill list
        hid, hl_t = torch.as_tensor(hist), torch.as_tensor(hl).to(torch.int32)
        s, p, g = sh._recommend_tiles(hid, hl_t, torch.arange(10), 4, 8, 2, 2, True, 1, 18, False)
        assert (s == float('-inf')).all() and (p == -1).all() and (g == -1).all()
        assert sh._recommend_tiles(hid, hl_t, torch.arange(10), 4, 8, 2, 2, True, None, None, False)[2] is None
        # the gathered rank lists are laid out [W, B, k] in rank order
        pool = np.arange(50)
        lists = []
        orig = sh._merge_rank_lists
        sh._merge_rank_lists = lambda *a: lists.append(a) or orig(*a)
        sh.recommend(hist, hl, pool, 6, False, 8, cuda_graph=False, max_per_category=2, collective=True)
        sh._merge_rank_lists = orig
        S, Pp, G, cap, groups = lists[0]
        assert S.shape == Pp.shape == G.shape == (world, 5, 6) and cap == 2 and groups == int(sh.cat.max()) + 1
        for r, (a, b) in enumerate(contiguous_blocks(7, world)[1]):
            mine = ref._recommend_tiles(hid, hl_t, torch.as_tensor(pool), 6, 8, a, b, False, 2, groups, False)
            assert torch.equal(S[r].view(torch.int32), mine[0].view(torch.int32)) and torch.equal(Pp[r], mine[1]) and torch.equal(G[r], mine[2]), r
        # every rank raises, naming the fields, when one rank is called with other inputs; the ranks stay in step
        pool = np.arange(50)
        with pytest.raises(RuntimeError, match=r'recommend.*k: \[5, 6'):
            sh.recommend(hist, hl, pool, 5 + (rank == 1), collective=True, cuda_graph=False)
        other = pool.copy()
        other[3] += rank == 1
        with pytest.raises(RuntimeError, match='pool_ids checksum') as err:
            sh.recommend(hist, hl, other, 5, collective=True, cuda_graph=False)
        assert 'k:' not in str(err.value)
        with pytest.raises(RuntimeError, match=r'max_per_category=|m: \[0, 2'):
            sh.recommend(hist, hl, pool, 5, collective=True, cuda_graph=False, max_per_category=None if rank == 0 else 2)
        # a check that fails on one rank only: RuntimeError everywhere, with that rank's reason on it
        with pytest.raises(RuntimeError, match='argument error') as err:
            sh.recommend(hist, hl, pool, 0 if rank == 1 else 5, collective=True, cuda_graph=False)
        assert ('k must be in' in str(err.value)) == (rank == 1)
        # a check that fails on every rank raises its ValueError on every rank
        with pytest.raises(ValueError, match='pool_tile must be'):
            sh.recommend(hist, hl, pool, 5, pool_tile=5000, collective=True, cuda_graph=False)
        got = sh.recommend(hist, hl, pool, 5, pool_tile=8, collective=True, cuda_graph=False)
        want = ref.recommend(hist, hl, pool, 5, pool_tile=8, cuda_graph=False)
        assert _same(got, want)
        q.put((rank, 'ok'))
    except BaseException as ex:
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        q.close()
        q.join_thread()
        os._exit(0)


@pytest.mark.parametrize('world', [2, 3, 4])
def test_collective_recommend_host_logic_equals_plain_scorer(world):
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        results = [q.get(timeout=300) for _ in range(world)]
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    for rank, msg in sorted(results):
        assert msg == 'ok', 'rank %d: %s' % (rank, msg)
