"""GPU tests of evaluation through the factored cluster tail (CorpusScorer.score / evaluate(exact=False),
nnr_cluster_tail_scores_packed).

  * the packed kernel against the float64 unfactored reference of tests.test_recommend_factored_gpu, per user: ragged
    lists with counts 0, 1, 37, 300 and more than one CTA slice, a history of padding only, one non-empty cluster,
    H = 256 with C1 = 72, D = 356, tiny sizes; entries past each count keep their NaN sentinel;
  * bit-equal to the pool kernel (nnr_cluster_tail_scores) when every user is given the same rows;
  * score(exact=False) against score() and the fp64 oracle for SUE, SUE_wo_GCN, SUE_wo_HCA (bit-equal there),
    gcn_layer_norm and every graph flag;
  * evaluate(exact=False) on a ragged set against the exact call: scores, ranks up to near ties, metrics, -1 padding,
    the same impressions padded to two widths;
  * deterministic, graph replay equals host launches, peak memory below one exact batch's tail buffers, and the NCCL
    collective equals the plain call.
"""
import math
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import nnr_oracle as O
from tests.test_recommend_factored_gpu import _reference, _tail_inputs
from tests.test_recommend_gpu import (NEWS, TOL, _build, _config, _corpus, _oracle_scores, _scorer,
                                      sue)  # noqa: F401  (sue: fixture)
from tests.test_scoring_dp_gloo import _free_port
from tests.util import rel_err

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.contiguous().cpu().view(torch.int32)


# ---- the kernel alone --------------------------------------------------------------------------------------------------
def _packed_inputs(counts, Hh, C1, D, Au, dev, seed):
    """the user side of _tail_inputs for len(counts) users, and each user's own candidate rows stored back to back"""
    B, R = len(counts), max(1, sum(counts))
    Kp, g, W, idx, cmask, Qp, qk2, cand, bias = _tail_inputs(B, Hh, C1, D, Au, R, dev, seed)
    row_off = torch.tensor([0] + list(np.cumsum(counts)), dtype=torch.int32, device=dev)
    return Kp, g, W, idx, cmask, Qp, qk2, cand, bias, row_off


def _run_packed(Kp, g, W, idx, cmask, Qp, qk2, cand, bias, row_off, n_max, scale, lds=None):
    from nnr_b200 import ops
    f = lambda x: x.float().contiguous()
    B, Hh, D = g.shape
    out = torch.full((B, lds or n_max), float('nan'), device=g.device)
    ops.cluster_tail_scores_packed(f(Kp), f(g), f(g @ W.T), idx, cmask.to(torch.uint8), row_off, f(Qp), f(qk2), f(cand),
                                   f(bias), B, Hh, Kp.shape[2], D, cmask.shape[1], n_max, scale, out)
    return out


@pytest.mark.parametrize('counts, Hh, C1, D, Au', [
    ([37, 0, 1, 300, 129, 37], 50, 19, 900, 225),      # the default model: empty, single, MIND-sized and long lists
    ([5, 64, 65, 0], 256, 72, 900, 225),               # the limits; 64 / 65 candidates: one and two 64-candidate slices
    ([20, 3, 77], 20, 19, 356, 200),                   # hidden_dim 64: D = 356
    ([1, 2, 3], 8, 5, 16, 3),                          # tiny sizes
])
def test_packed_kernel_matches_float64_reference(cuda, counts, Hh, C1, D, Au):
    args = _packed_inputs(counts, Hh, C1, D, Au, cuda, seed=sum(counts) + Hh)
    Kp, g, W, idx, cmask, Qp, qk2, cand, bias, row_off = args
    n_max, scale = max(counts), 1.0 / math.sqrt(Au)
    got = _run_packed(*args, n_max, scale, lds=n_max + 3)
    for b, c in enumerate(counts):
        assert torch.isnan(got[b, c:]).all(), b                                         # past the count: not written
        if c == 0:
            continue
        r = slice(int(row_off[b]), int(row_off[b + 1]))
        ref = _reference(Kp[b:b + 1], g[b:b + 1], W, idx[b:b + 1], cmask[b:b + 1], Qp[r], qk2[r], cand[r], bias, scale)[0]
        assert rel_err(got[b, :c], ref) <= 1e-5, (b, rel_err(got[b, :c], ref))


def test_packed_kernel_clamps_bad_offsets(cuda):
    """offsets past the rows, decreasing and beyond n_max are clamped: nothing is read or written out of bounds"""
    args = _packed_inputs([10, 10, 10], 50, 19, 900, 225, cuda, seed=5)
    *user, Qp, qk2, cand, bias, _ = args
    good = _run_packed(*user, Qp, qk2, cand, bias, torch.tensor([0, 10, 20, 30], dtype=torch.int32, device=cuda), 10, 0.1)
    bad = _run_packed(*user, Qp, qk2, cand, bias, torch.tensor([0, 25, 5, 10 ** 6], dtype=torch.int32, device=cuda), 8, 0.1)
    torch.cuda.synchronize()
    assert torch.equal(_bits(bad[0, :8]), _bits(good[0, :8]))                          # count 25 clamped to n_max = 8
    assert torch.isnan(bad[1]).all()                                                   # a decreasing offset: count 0
    assert not torch.isnan(bad[2, :8]).any()                                           # rows [5, 30): clamped to the rows


@pytest.mark.parametrize('B, Hh, C1, D, Au, T', [
    (4, 50, 19, 900, 225, 37),
    (3, 50, 19, 900, 225, 300),
    (2, 256, 72, 900, 225, 130),
    (3, 20, 19, 356, 200, 65),
])
def test_packed_kernel_equals_pool_kernel_bit_for_bit(cuda, B, Hh, C1, D, Au, T):
    from nnr_b200 import ops
    Kp, g, W, idx, cmask, Qp, qk2, cand, bias = _tail_inputs(B, Hh, C1, D, Au, T, cuda, seed=T)
    f = lambda x: x.float().contiguous()
    Wg, scale = f(g @ W.T), 1.0 / math.sqrt(Au)
    pool = torch.empty(B, T, device=cuda)
    ops.cluster_tail_scores(f(Kp), f(g), Wg, idx, cmask.to(torch.uint8), f(Qp), f(qk2), f(cand), f(bias), B, Hh, Au, D, C1,
                            T, scale, pool)
    rows = lambda x: f(x).repeat(B, 1)                                                 # every user gets the same T rows
    row_off = torch.arange(B + 1, dtype=torch.int32, device=cuda) * T
    packed = torch.empty(B, T, device=cuda)
    ops.cluster_tail_scores_packed(f(Kp), f(g), Wg, idx, cmask.to(torch.uint8), row_off, rows(Qp), rows(qk2), rows(cand),
                                   f(bias), B, Hh, Au, D, C1, T, scale, packed)
    assert torch.equal(_bits(packed), _bits(pool))


# ---- score(exact=False) ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kw', [dict(user_encoder='SUE'), dict(user_encoder='SUE_wo_HCA'), dict(user_encoder='SUE_wo_GCN'),
                                dict(gcn_layer_norm=True)], ids=['SUE', 'SUE_wo_HCA', 'SUE_wo_GCN', 'layer_norm'])
def test_factored_score_matches_exact_and_oracle(cuda, kw):
    cfg = _config(**kw)
    p = O.formula_params(cfg)
    syn = _corpus()
    sc = _scorer(_build(cfg, p, cuda), syn)
    pool = np.random.default_rng(9).permutation(NEWS)[:70]
    for B in (6, 70):                                                                  # eager and graphed
        hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=4 + B)
        cand = np.tile(pool, (B, 1))
        got, exact = sc.score(hist, hl, cand, exact=False), sc.score(hist, hl, cand)
        assert rel_err(got, exact) <= 1e-4
        assert rel_err(got.cpu(), _oracle_scores(p, cfg, syn, hist, hl, pool)) < TOL
        if kw.get('user_encoder') == 'SUE_wo_HCA':                                     # no candidate-dependent tail
            assert torch.equal(_bits(got), _bits(exact))


def test_factored_score_with_graph_flags_matches_oracle(sue, cuda):
    from nnr_b200 import ops
    from tests.test_pins import FLAG_SETS
    _, syn, p, cfg = sue
    m = _build(cfg, p, cuda)
    hist, hl, _ = syn.sample_behaviors(6, news_num=1, seed=8)
    pool = np.random.default_rng(3).permutation(NEWS)[:50]
    for flags in FLAG_SETS:
        sc = _scorer(m, syn, graph_flags=ops.graph_flags(**flags))
        got = sc.score(hist, hl, np.tile(pool, (6, 1)), exact=False).cpu()
        assert rel_err(got, _oracle_scores(p, cfg, syn, hist, hl, pool, flags)) < TOL, flags


# ---- evaluate(exact=False) on a ragged set -----------------------------------------------------------------------------
def _ragged(syn, I, n_max, seed, pad=-1):
    """I impressions with long-tailed counts in [1, n_max] (some at n_max), one positive each, padding ids ``pad``"""
    rng = np.random.default_rng(seed)
    hist, hl, _ = syn.sample_behaviors(I, news_num=1, seed=seed)
    cnt = np.minimum(n_max, np.maximum(2, rng.lognormal(2.5, 0.9, I).astype(np.int64)))
    cnt[:3] = n_max
    cand = rng.integers(0, NEWS, (I, n_max))
    valid = np.arange(n_max)[None, :] < cnt[:, None]
    cand = np.where(valid, cand, pad)
    lab = np.zeros((I, n_max), dtype=np.int64)
    lab[np.arange(I), rng.integers(0, cnt)] = 1
    return hist, hl, cand, cnt, lab, valid


def test_factored_evaluate_on_a_ragged_set(sue):
    sc, syn, _, _ = sue
    hist, hl, cand, cnt, lab, valid = _ragged(syn, 300, 120, seed=7)
    *m_f, r_f = sc.evaluate(hist, hl, cand, cnt, lab, batch=128, exact=False)
    S = sc._impression_scores(hist, hl, np.where(valid, cand, 0), 128).cpu()           # the exact scores
    F = sc._impression_scores(hist, hl, cand, 128, cnt, lab, exact=False).cpu()
    v = torch.from_numpy(valid)
    assert rel_err(F[v], S[v]) <= 1e-4
    *m_e, r_e = sc.evaluate(hist, hl, np.where(valid, cand, 0), cnt, lab, batch=128)
    tol = 1e-4 * S[v].abs().max().item()
    diff = (r_f.cpu() != r_e.cpu())
    for i in torch.nonzero(diff.any(1)).flatten().tolist():                            # ranks differ only between near ties
        c = int(cnt[i])
        for j in torch.nonzero(diff[i, :c]).flatten().tolist():
            rf = int(r_f[i, j])
            other = int(torch.nonzero(r_e[i, :c].cpu() == rf)[0])
            assert abs(S[i, j] - S[i, other]) <= 2 * tol, (i, j, other)
    if not diff.any():                                                                 # the seeded set: no near tie
        assert m_f == m_e
    assert np.allclose(m_f, m_e, rtol=0, atol=1e-3), (m_f, m_e)
    assert (r_f.cpu()[~v] == 0).all()


def test_factored_evaluate_is_independent_of_the_padding_width(sue):
    sc, syn, _, _ = sue
    hist, hl, cand, cnt, lab, valid = _ragged(syn, 150, 37, seed=3)
    wide_c = np.full((150, 300), -1)
    wide_c[:, :37] = cand
    wide_l = np.zeros((150, 300), dtype=np.int64)
    wide_l[:, :37] = lab
    *m_n, r_n = sc.evaluate(hist, hl, cand, cnt, lab, batch=64, exact=False)
    *m_w, r_w = sc.evaluate(hist, hl, wide_c, cnt, wide_l, batch=64, exact=False)
    assert torch.equal(r_w[:, :37].cpu(), r_n.cpu()) and (r_w[:, 37:] == 0).all()
    assert np.allclose(m_w, m_n, rtol=1e-12, atol=0), (m_w, m_n)
    s_n = sc._impression_scores(hist, hl, cand, 64, cnt, lab, exact=False).cpu()
    s_w = sc._impression_scores(hist, hl, wide_c, 64, cnt, wide_l, exact=False).cpu()[:, :37]
    v = torch.from_numpy(valid)
    assert rel_err(s_w[v], s_n[v]) <= 1e-6


def test_factored_evaluate_is_deterministic_and_graph_replay_equals_host_launch(sue):
    sc, syn, _, _ = sue
    hist, hl, cand, cnt, lab, valid = _ragged(syn, 200, 60, seed=11)
    a = sc._impression_scores(hist, hl, cand, 64, cnt, lab, exact=False)               # 3 graphed batches + a short one
    assert ('score_factored', (64, hist.shape[1]), (64, 60), sc.cache.data_ptr()) in sc._graphs
    b = sc._impression_scores(hist, hl, cand, 64, cnt, lab, exact=False)
    v = torch.from_numpy(valid)
    eager = torch.cat([sc._score_packed(hist[s:s + 64], hl[s:s + 64], torch.from_numpy(cand[s:s + 64]),
                                        torch.from_numpy(cnt[s:s + 64]), False) for s in range(0, 200, 64)])
    assert torch.equal(_bits(a), _bits(b)) and torch.equal(_bits(a.cpu()[v]), _bits(eager.cpu()[v]))
    ra, rb = sc.evaluate(hist, hl, cand, cnt, lab, batch=64, exact=False), sc.evaluate(hist, hl, cand, cnt, lab, batch=64,
                                                                                       exact=False)
    assert ra[:4] == rb[:4] and torch.equal(ra[4], rb[4])
    s1 = sc.score(hist[:70], hl[:70], np.where(valid, cand, 0)[:70], exact=False)      # score(): graph vs host launch
    s2 = sc.score(hist[:70], hl[:70], np.where(valid, cand, 0)[:70], exact=False, cuda_graph=False)
    assert torch.equal(_bits(s1), _bits(s2))


def test_factored_evaluate_peak_memory_is_below_one_exact_batch_tail(sue):
    sc, syn, _, _ = sue
    B, n_max = 64, 300
    hist, hl, cand, cnt, lab, _ = _ragged(syn, B, n_max, seed=13)
    sc._graphs.pop(('score_factored', (B, hist.shape[1]), (B, n_max), sc.cache.data_ptr()), None)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    sc.evaluate(hist, hl, cand, cnt, lab, batch=B, exact=False)                       # with the graph's capture and pool
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    D, C1 = sc.cache.shape[1], sc._category_num() + 1
    tail = 4 * B * n_max * C1 * D * 4                                                  # the exact tail's four fp32 buffers
    assert peak < tail, (peak, tail)


# ---- collective ------------------------------------------------------------------------------------------------------
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
        hist, hl, cand, cnt, lab, _ = _ragged(syn, 150, 80, seed=31)
        *m_r, r_r = ref.evaluate(hist, hl, cand, cnt, lab, batch=32, exact=False)
        *m_s, r_s = sh.evaluate(hist, hl, cand, cnt, lab, batch=32, exact=False)
        assert m_r == m_s and torch.equal(r_r, r_s)
        if world > 1:                                          # ranks that disagree on exact all raise
            with pytest.raises(RuntimeError, match='exact'):
                sh.evaluate(hist, hl, np.maximum(cand, 0), cnt, lab, batch=32, exact=rank == 0)
        bad = cnt.copy()
        bad[0] = 81
        with pytest.raises(ValueError, match='candidate_count'):                       # the same bad input on every rank
            sh.evaluate(hist, hl, cand, bad, lab, batch=32, exact=False)
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


@pytest.mark.parametrize('world', [1, 2])
def test_factored_evaluate_collective_equals_plain_call(world):
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
