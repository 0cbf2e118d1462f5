"""GPU tests of the data-parallel CorpusScorer over NCCL: with a process group, ``encode_corpus`` and ``evaluate`` share the
corpus chunks and the impression batches between the ranks and all-gather the results.  Every rank must get exactly what
the plain single-GPU scorer computes on its own device: the same cache, scores, ranks and metrics, compared bit for bit.

The cases: a corpus whose chunk count is not a multiple of the world size, with a partial last chunk (5 chunks of 64,
the graph path included); a corpus with fewer chunks than ranks; impression counts that are not a multiple of the batch,
and fewer than batch x world, so that some rank scores nothing; candidate counts that vary, including 0.  And the input
check: a rank called with a different impression count makes every rank raise instead of entering the all-gather.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

BATCH = 64


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _impressions(syn, n_imp, seed):
    """history ids / lengths, [n_imp, 6] candidates 0-padded past a count in {0, 2, ..., 6}, one positive per impression"""
    hist, hl, cand = syn.sample_behaviors(n_imp, news_num=6, seed=seed)
    rng = np.random.default_rng(seed)
    cnt = rng.choice([0, 2, 3, 4, 5, 6], size=n_imp)
    cnt[0], cnt[-1] = 0, 6
    lab = np.zeros(cand.shape, dtype=np.int64)
    for b in range(n_imp):
        cand[b, cnt[b]:] = 0
        if cnt[b]:
            lab[b, rng.integers(0, cnt[b])] = 1
    return hist, hl, cand, cnt, lab


def _worker(rank, world, port, q, case):
    try:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        torch.cuda.set_device(rank)
        dev = torch.device('cuda', rank)
        dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
        import nnr_b200
        from nnr_b200 import engine
        from nnr_b200.scoring import CorpusScorer
        from nnr_b200.synthetic import SyntheticMIND
        from oracle import nnr_oracle as O
        engine.sort_fn = O.stable_sort
        cfg = O.make_config(vocabulary_size=600, max_history_num=8, max_title_length=10, max_abstract_length=20,
                            subCategory_num=30, gcn_layer_num=2)
        p = O.formula_params(cfg)
        cfg.pretrained_word_embedding = p['news_encoder.word_embedding.weight']
        m = nnr_b200.Model(cfg)
        m.initialize()
        m.load_state_dict(O.alias_state_dict(p))
        m.to(dev).eval()
        group = dist.group.WORLD

        def corpus(news_num):
            syn = SyntheticMIND(news_num=news_num, vocabulary_size=600, subCategory_num=30, max_title_length=10,
                                max_abstract_length=20, max_history_num=8, lengths='mind', seed=23)
            fields = (syn.news_title_text, syn.news_title_mask, syn.news_abstract_text, syn.news_abstract_mask,
                      syn.news_category, syn.news_subCategory)
            return syn, fields

        if case == 'equal':
            # 300 news = 4 full chunks of 64 + 44 (graph path for the full ones); 44 news = 1 chunk, 172 = 3 chunks
            for news_num in (300, max(44, 64 * (world - 1) - 20)):
                syn, fields = corpus(news_num)
                ref = CorpusScorer(m, *fields, chunk=64)
                sh = CorpusScorer(m, *fields, chunk=64, process_group=group)
                cache = sh.encode_corpus()
                assert torch.equal(cache, ref.encode_corpus()), ('cache', news_num)
                for n_imp in (150, 40):                      # 3 batches of 64 (the last one partial), 1 partial batch
                    hist, hl, cand, cnt, lab = _impressions(syn, n_imp, seed=news_num + n_imp)
                    s_sh = sh._impression_scores(hist, hl, cand, BATCH, cnt, lab)
                    s_ref = ref._impression_scores(hist, hl, cand, BATCH)
                    assert s_sh.shape == (n_imp, 6) and torch.equal(s_sh, s_ref), ('scores', news_num, n_imp)
                    *m_sh, r_sh = sh.evaluate(hist, hl, cand, cnt, lab, batch=BATCH)
                    *m_ref, r_ref = ref.evaluate(hist, hl, cand, cnt, lab, batch=BATCH)
                    assert torch.equal(r_sh, r_ref), ('ranks', news_num, n_imp)
                    assert m_sh == m_ref and all(np.isfinite(m_ref)), ('metrics', news_num, n_imp, m_sh, m_ref)
                if rank == 0:                                 # score() is rank-local: the other ranks do not join it
                    hist, hl, cand = syn.sample_behaviors(BATCH, news_num=5, seed=1)
                    assert torch.equal(sh.score(hist, hl, cand), ref.score(hist, hl, cand))
                dist.barrier()
        else:
            syn, fields = corpus(300)
            sh = CorpusScorer(m, *fields, chunk=64, process_group=group)
            sh.encode_corpus()
            hist, hl, cand, cnt, lab = _impressions(syn, 150, seed=3)
            n_imp = 150 - rank                               # rank 1 passes one impression less
            try:
                sh.evaluate(hist[:n_imp], hl[:n_imp], cand[:n_imp], cnt[:n_imp], lab[:n_imp], batch=BATCH)
                raise AssertionError('evaluate() with different inputs on the ranks did not raise')
            except RuntimeError as ex:
                assert 'I: [150, 149]' in str(ex), str(ex)
            # the ranks stay in step after the rejected call
            *_, ranks = sh.evaluate(hist, hl, cand, cnt, lab, batch=BATCH)
            assert ranks.shape == (150, 6)
            if rank == 1:                                     # a model that is not on the current device is rejected
                torch.cuda.set_device(0)
                with pytest.raises(RuntimeError, match='current CUDA device'):
                    CorpusScorer(m, *fields, chunk=64, process_group=group)
                torch.cuda.set_device(1)
        torch.cuda.synchronize()
        q.put((rank, 'ok'))
    except BaseException as ex:                               # surface the failure in the parent
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        # no destroy_process_group(): the worker process ends here anyway
        import sys
        sys.stdout.flush()
        q.close()
        q.join_thread()                                        # the result must reach the parent before the hard exit
        os._exit(0)


def _run(world, case):
    if torch.cuda.device_count() < world:
        pytest.skip('needs %d GPUs' % world)
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


def test_group_of_one_rank_equals_plain_scorer():
    _run(1, 'equal')


@pytest.mark.parametrize('world', [2, 4])
def test_sharded_scorer_equals_one_gpu(world):
    _run(world, 'equal')


def test_ranks_called_with_different_inputs_all_raise():
    _run(2, 'mismatch')
