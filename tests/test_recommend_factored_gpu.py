"""GPU tests of top-k recommendation through the factored cluster tail (CorpusScorer.recommend(exact=False),
nnr_cluster_tail_scores).

  * the kernel against a float64 torch reference of the formula computed the unfactored way (intra-cluster features, the
    affine on them, relu, residual, masked inter-cluster softmax, dot): empty clusters, a history of padding only, one
    non-empty cluster, H = 256 with C1 = 72, T = 1, odd T and T = 4096, D = 900 and D = 356;
  * recommend(exact=False) against the fp64 oracle for SUE, SUE_wo_GCN, SUE_wo_HCA, gcn_layer_norm and every graph flag;
  * against the exact path: scores within 1e-4 of score(), ids equal except near the k-th score, and the result is the
    stated order (tests.test_recommend_gpu.stated_order) / the capped greedy rule of the factored scores themselves;
  * deterministic, graph replay equals host launches, the collective equals the plain call, memory does not grow with P.
"""
import math
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import nnr_oracle as O
from tests.test_recommend_capped_gpu import _eligible, capped_reference
from tests.test_recommend_gpu import (H, NEWS, TOL, _build, _config, _corpus, _oracle_scores, _scorer, stated_order,
                                      sue, tiled_scores)  # noqa: F401  (sue: fixture)
from tests.test_scoring_dp_gloo import _free_port
from tests.util import rel_err

pytestmark = pytest.mark.gpu


def _same(a, b):
    """ids equal and scores equal bit for bit"""
    return torch.equal(a[0].cpu(), b[0].cpu()) and torch.equal(a[1].cpu().view(torch.int32), b[1].cpu().view(torch.int32))


# ---- the kernel alone --------------------------------------------------------------------------------------------------
def _reference(Kp, g, W, idx, cmask, Qp, qk2, cand, bias, scale):
    """float64, unfactored: intra[b,t,c] = sum_{h in c} alpha g_h, f = relu(W intra + b) + intra, beta = masked softmax of
    scale * f.qk2, score = sum_c beta f.cand"""
    B, Hh, D = g.shape
    C1 = cmask.shape[1]
    idx = idx.clamp(0, C1 - 1)
    onehot = torch.nn.functional.one_hot(idx, C1).to(torch.float64)                        # [B, H, C1]
    s = scale * torch.einsum('bha,ta->bth', Kp, Qp)                                         # [B, T, H]
    same = onehot @ onehot.transpose(1, 2)                                                  # [B, H, H]: same cluster
    m = torch.where(same[:, None] > 0, s[:, :, None, :], torch.tensor(-math.inf, dtype=s.dtype, device=s.device)).amax(3)
    e = torch.exp(s - m)
    alpha = e / torch.einsum('bth,bkh->btk', e, same)                                       # segment softmax
    out = []
    for t0 in range(0, Qp.shape[0], 256):                                                   # [B, 256, C1, D] at a time
        a = alpha[:, t0:t0 + 256]
        intra = torch.einsum('bth,bhc,bhd->btcd', a, onehot, g)
        f = torch.relu(intra @ W.T + bias) + intra
        lq = scale * torch.einsum('btcd,td->btc', f, qk2[t0:t0 + 256])
        lq = torch.where(cmask[:, None, :] > 0, lq, torch.tensor(-1e9, dtype=lq.dtype, device=lq.device))
        beta = torch.softmax(lq, 2)
        out.append(torch.einsum('btc,btcd,td->bt', beta, f, cand[t0:t0 + 256]))
    return torch.cat(out, 1)


def _tail_inputs(B, Hh, C1, D, Au, T, dev, seed):
    gen = torch.Generator().manual_seed(seed)
    r = lambda *shape, s=1.0: (torch.randn(*shape, generator=gen, dtype=torch.float64) * s).to(dev)
    Kp, Qp = r(B, Hh, Au), r(T, Au)
    g, qk2, cand = r(B, Hh, D, s=0.5), r(T, D, s=0.5), r(T, D, s=0.5)
    W, bias = r(D, D, s=1.0 / math.sqrt(D)), r(D, s=0.3)
    idx = torch.randint(0, C1, (B, Hh), generator=gen)
    idx[0, ::3] = torch.randint(0, max(1, C1 // 3), (len(range(0, Hh, 3)),), generator=gen)   # user 0: skewed, empty clusters
    idx[0, 1], idx[0, 2] = -3, C1 + 5                                                    # clamped like cluster_intra_fwd
    cmask = torch.rand(B, C1, generator=gen) < 0.6
    if B > 1:                                                                            # user 1: a history of padding only
        idx[1] = C1 - 1
        cmask[1] = False
    if B > 2:                                                                            # user 2: one non-empty cluster
        idx[2] = min(3, C1 - 1)
        cmask[2] = False
        cmask[2, min(3, C1 - 1)] = True
    cmask[:, -1] = True                                                                  # encode_user: cluster C unmasked
    return Kp, g, W, idx.to(dev), cmask.to(dev), Qp, qk2, cand, bias


def _run_tail(Kp, g, W, idx, cmask, Qp, qk2, cand, bias, scale, lds=None):
    from nnr_b200 import ops
    f = lambda x: x.float().contiguous()
    B, Hh, D = g.shape
    T = Qp.shape[0]
    Wg = g @ W.T                                                                          # the user side's Wg, in fp64
    out = torch.full((B, lds or T), float('nan'), device=g.device)
    scores = out[:, :T]
    ops.cluster_tail_scores(f(Kp), f(g), f(Wg), idx, cmask.to(torch.uint8), f(Qp), f(qk2), f(cand), f(bias), B, Hh,
                            Kp.shape[2], D, cmask.shape[1], T, scale, scores)
    return out


@pytest.mark.parametrize('B, Hh, C1, D, Au, T', [
    (3, 50, 19, 900, 225, 1),          # the default model, one candidate
    (4, 50, 19, 900, 225, 333),        # odd T: a partial CTA
    (2, 256, 72, 900, 225, 4096),      # the limits: the 128-candidate CTA, T at the tile limit
    (5, 20, 19, 356, 200, 257),        # hidden_dim 64: D = 356
    (3, 8, 5, 16, 3, 130),             # tiny sizes: Au below one staged chunk, D = two feature steps
])
def test_tail_kernel_matches_float64_reference(cuda, B, Hh, C1, D, Au, T):
    args = _tail_inputs(B, Hh, C1, D, Au, T, cuda, seed=B + Hh + T)
    scale = 1.0 / math.sqrt(Au)
    got = _run_tail(*args, scale, lds=T + 3)
    assert torch.isnan(got[:, T:]).all()                                                 # the row stride is honoured
    ref = _reference(*args, scale)
    err = rel_err(got[:, :T], ref)
    assert err <= 1e-5, err
    for b in range(B):                                                                   # every user, not just the largest
        assert rel_err(got[b, :T], ref[b]) <= 1e-5 * ref.abs().max().item() / ref[b].abs().max().item(), b


def test_tail_kernel_is_deterministic(cuda):
    args = _tail_inputs(6, 50, 19, 900, 225, 700, cuda, seed=3)
    a, b = _run_tail(*args, 0.0667), _run_tail(*args, 0.0667)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


# ---- recommend(exact=False) against the oracle ---------------------------------------------------------------------
def _factored_all(sc, hist, hl, pool, T):
    """every pool entry's score from recommend(exact=False) (k = P, no exclusion), back in pool order (distinct pool ids)"""
    ids, scores = sc.recommend(hist, hl, pool, len(pool), exclude_history=False, pool_tile=T, exact=False)
    where = {int(i): j for j, i in enumerate(pool)}
    out = torch.empty(len(hl), len(pool))
    for b in range(len(hl)):
        out[b, [where[int(i)] for i in ids[b]]] = scores[b].cpu()
    return out


@pytest.mark.parametrize('kw', [dict(user_encoder='SUE'), dict(user_encoder='SUE_wo_HCA'), dict(user_encoder='SUE_wo_GCN'),
                                dict(gcn_layer_norm=True)], ids=['SUE', 'SUE_wo_HCA', 'SUE_wo_GCN', 'layer_norm'])
def test_factored_scores_match_oracle(cuda, kw):
    cfg = _config(**kw)
    p = O.formula_params(cfg)
    syn = _corpus()
    sc = _scorer(_build(cfg, p, cuda), syn)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=4)
    pool = np.random.default_rng(9).permutation(NEWS)[:70]
    assert rel_err(_factored_all(sc, hist, hl, pool, 32), _oracle_scores(p, cfg, syn, hist, hl, pool)) < TOL
    if kw.get('user_encoder') == 'SUE_wo_HCA':          # the user vector does not depend on the candidate: the exact path
        for T in (32, 70):
            assert _same(sc.recommend(hist, hl, pool, 20, pool_tile=T, exact=False), sc.recommend(hist, hl, pool, 20, pool_tile=T))


def test_factored_scores_with_graph_flags_match_oracle(sue, cuda):
    from nnr_b200 import ops
    from tests.test_pins import FLAG_SETS
    _, syn, p, cfg = sue
    m = _build(cfg, p, cuda)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=8)
    pool = np.random.default_rng(3).permutation(NEWS)[:50]
    for flags in FLAG_SETS:
        sc = _scorer(m, syn, graph_flags=ops.graph_flags(**flags))
        assert rel_err(_factored_all(sc, hist, hl, pool, 32), _oracle_scores(p, cfg, syn, hist, hl, pool, flags)) < TOL, flags


# ---- against the exact path --------------------------------------------------------------------------------------------
@pytest.mark.parametrize('B, P, T, k, exclude', [
    (6, 150, 64, 10, True),         # P not a multiple of T: two graphed tiles and an eager one
    (6, 150, 64, 10, False),
    (6, 150, 32, 1024, True),       # k above the eligible entries: fill
    (1, 150, 16, 20, True),         # one user
    (70, 100, 32, 12, True),        # B >= 64
    (6, 150, None, 25, True),       # the default tile: the whole pool
])
def test_factored_recommend_against_the_exact_path(sue, B, P, T, k, exclude):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=B + P + k)
    pool = np.random.default_rng(P + k).permutation(NEWS)[:P]
    Tt = T or P
    S = tiled_scores(sc, hist, hl, pool, Tt).cpu()                                    # score() of every pool entry
    F = _factored_all(sc, hist, hl, pool, Tt)
    assert rel_err(F, S) <= 1e-4
    # the result is the stated order of the factored scores themselves
    ids, scores = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T, exact=False)
    rid, rscore = stated_order(F, pool, hist, hl, k, exclude)
    assert torch.equal(ids.cpu(), rid) and torch.equal(scores.cpu(), rscore)
    # and equals the exact path's ids except near the k-th exact score
    eid, _ = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T)
    tol = 1e-4 * S.abs().max().item()
    where = {int(i): j for j, i in enumerate(pool)}
    for b in range(B):
        got, want = ids[b].cpu().tolist(), eid[b].cpu().tolist()
        real = [i for i in want if i >= 0]
        kth = S[b, where[real[-1]]].item() if len(real) == k else -math.inf
        for i in set(got) ^ set(want):
            assert i >= 0 and abs(S[b, where[i]].item() - kth) <= tol, (b, i)
        ex = [S[b, where[i]].item() for i in got if i >= 0]
        assert all(y <= x + 2 * tol for x, y in zip(ex, ex[1:])), b                 # best first, up to near ties
        assert sum(i < 0 for i in got) == sum(i < 0 for i in want)                   # the same fill


@pytest.mark.parametrize('m', [1, 2])
def test_factored_capped_recommend_equals_greedy_reference(sue, m):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(5, news_num=1, seed=17)
    cats = syn.news_category
    big = int(np.bincount(cats).argmax())
    rng = np.random.default_rng(6)
    own = np.flatnonzero(cats == big)                                   # distinct ids: _factored_all maps ids to positions
    pool = rng.permutation(np.concatenate([own, rng.choice(np.flatnonzero(cats != big), len(own) // 2, replace=False)]))
    T, k = 16, 12
    F = _factored_all(sc, hist, hl, pool, T).numpy()
    for exclude in (False, True):
        ids, scores = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T, max_per_category=m, exact=False)
        rs, rp, _ = capped_reference(F, cats[pool], _eligible(pool, hist, hl, exclude), k, m)
        assert np.array_equal(ids.cpu().numpy(), np.where(rp >= 0, pool[np.maximum(rp, 0)], -1))
        assert np.array_equal(scores.cpu().numpy(), rs)


def test_factored_recommend_is_deterministic_and_graph_replay_equals_host_launch(sue):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(9, news_num=1, seed=11)
    pool = np.random.default_rng(2).permutation(NEWS)[:140]
    eager = sc.recommend(hist, hl, pool, 25, pool_tile=32, cuda_graph=False, exact=False)
    graphed = sc.recommend(hist, hl, pool, 25, pool_tile=32, exact=False)
    assert ('recommend_factored', 9, H, 32, sc.cache.data_ptr()) in sc._graphs
    again = sc.recommend(hist, hl, pool, 25, pool_tile=32, exact=False)
    eager2 = sc.recommend(hist, hl, pool, 25, pool_tile=32, cuda_graph=False, exact=False)
    for other in (graphed, again, eager2):
        assert _same(eager, other)
    hist2, hl2, _ = syn.sample_behaviors(9, news_num=1, seed=12)                   # replays with another user side
    assert _same(sc.recommend(hist2, hl2, pool, 25, pool_tile=32, exact=False),
                 sc.recommend(hist2, hl2, pool, 25, pool_tile=32, cuda_graph=False, exact=False))


@pytest.mark.parametrize('cuda_graph', [False, True])
def test_factored_recommend_memory_does_not_grow_with_the_pool(sue, cuda_graph):
    sc, syn, _, _ = sue
    B, T = 32, 64
    hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=13)
    pool = torch.from_numpy(np.random.default_rng(4).integers(0, NEWS, 8 * T))

    def peak(P):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        sc.recommend(hist, hl, pool[:P], 10, pool_tile=T, cuda_graph=cuda_graph, exact=False)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base
    peak(T), peak(8 * T)                                                 # warm-up: graph capture, workspaces
    one, eight = peak(T), peak(8 * T)
    assert eight <= 1.03 * one + 65536, (one, eight)


# ---- collective ------------------------------------------------------------------------------------------------------
def _simulated_collective(sc, hist, hl, pool, k, T, W, exclude=True, m=None):
    """recommend(collective=True, exact=False) over W ranks, on one device: every rank's list, then the final merge"""
    from nnr_b200.scoring import contiguous_blocks
    hid, hl_, pool_, k, T, m_, groups = sc._recommend_inputs(hist, hl, pool, k, exclude, T, m, exact=False)
    parts = contiguous_blocks(-(-pool_.numel() // T), W)[1]
    lists = [sc._recommend_tiles(hid, hl_, pool_, k, T, a, b, exclude, m_, groups, True, exact=False) for a, b in parts]
    S, P = torch.stack([x[0] for x in lists]), torch.stack([x[1] for x in lists])
    G = torch.stack([x[2] for x in lists]) if m_ is not None else None
    best_s, best_p = sc._merge_rank_lists(S, P, G, m_, groups)
    return sc._pool_ids(pool_, best_p), best_s


@pytest.mark.parametrize('P, T, k, m, exclude', [
    (150, 64, 10, None, True),      # 3 tiles: a rank without tiles at W = 4
    (150, 16, 10, 2, True),
    (150, 32, 1024, None, False),   # fill
])
def test_factored_simulated_ranks_equal_plain_recommend(sue, P, T, k, m, exclude):
    sc, syn, _, _ = sue
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=P + T)
    pool = np.random.default_rng(P + T).permutation(NEWS)[:P]
    want = sc.recommend(hist, hl, pool, k, exclude_history=exclude, pool_tile=T, max_per_category=m, exact=False)
    for W in (2, 3, 4):
        assert _same(_simulated_collective(sc, hist, hl, pool, k, T, W, exclude, m), want), W


def _worker(rank, world, port, q):
    try:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        torch.cuda.set_device(rank)
        dev = torch.device('cuda', rank)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
        cfg = _config()
        m = _build(cfg, O.formula_params(cfg), dev)
        syn = _corpus()
        ref = _scorer(m, syn)
        sh = _scorer(m, syn, process_group=dist.group.WORLD)
        hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=31)
        for P, T, k, cap, exclude in [(150, 64, 10, None, True), (150, 16, 10, 1, True), (150, 32, 1024, 2, False),
                                      (150, None, 20, None, True)]:
            pool = np.random.default_rng(P + k).permutation(NEWS)[:P]
            want = ref.recommend(hist, hl, pool, k, exclude, T, max_per_category=cap, exact=False)
            got = sh.recommend(hist, hl, pool, k, exclude, T, max_per_category=cap, collective=True, exact=False)
            assert _same(got, want), (P, T, k, cap, exclude)
        if world > 1:                                          # ranks that disagree on exact all raise
            with pytest.raises(RuntimeError, match='exact'):
                sh.recommend(hist, hl, np.arange(100), 10, pool_tile=16, collective=True, exact=rank == 0)
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


def _run(world):
    if not torch.cuda.is_available() or torch.cuda.device_count() < world:
        pytest.skip('needs %d GPUs, found %d' % (world, torch.cuda.device_count() if torch.cuda.is_available() else 0))
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
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


@pytest.mark.parametrize('world', [1, 2, 4])
def test_factored_collective_equals_plain_recommend(world):
    _run(world)
