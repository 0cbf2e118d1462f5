"""CPU test of the data-parallel CorpusScorer's host logic over gloo, world sizes 2, 3 and 4: chunk and batch partition,
zero-padded send blocks, the all-gathers and the input-agreement check.  The CUDA encoders are replaced by fakes whose
output depends on the whole chunk they are called with (as the selective gate's pairing does), so a moved chunk boundary
changes the cache.  The sharded results must equal the plain scorer's bit for bit.  tests/test_scoring_dp_gpu.py runs the
real model over NCCL."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

BATCH = 64


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


class _Encoder(torch.nn.Module):
    news_embedding_dim = 4

    def forward(self, tt, tm, _a, ct, cm, _b, cat, sub, _c):
        x = torch.stack([tt[0].float().sum(1), ct[0].float().sum(1), cat[0].float(), sub[0].float()], 1)
        return (x + x.mean(0))[None]


class _Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.news_encoder = _Encoder()
        self.w = torch.nn.Parameter(torch.zeros(1))


def _scorer_class():
    from nnr_b200.scoring import CorpusScorer

    class CpuScorer(CorpusScorer):
        def _check_group(self):                               # gloo and CPU tensors: the host logic only
            pass

        def score(self, history_ids, history_len, candidate_ids, cuda_graph=True):
            hid, cid = torch.as_tensor(history_ids).long(), torch.as_tensor(candidate_ids).long()
            user = self.cache[hid].sum(1) + torch.as_tensor(history_len)[:, None].float()
            return (self.cache[cid] * user[:, None, :]).sum(2)
    return CpuScorer


def _corpus(n, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(0, 50, (n, 4), generator=g), torch.ones(n, 4), torch.randint(0, 50, (n, 5), generator=g),
            torch.ones(n, 5), torch.randint(0, 18, (n,), generator=g), torch.randint(0, 30, (n,), generator=g))


def _impressions(n_news, n_imp, seed):
    rng = np.random.default_rng(seed)
    hist = rng.integers(0, n_news, size=(n_imp, 8))
    hl = rng.integers(0, 9, size=n_imp)
    cand = rng.integers(0, n_news, size=(n_imp, 6))
    cnt = rng.choice([0, 2, 3, 4, 5, 6], size=n_imp)
    lab = np.zeros(cand.shape, dtype=np.int64)
    for b in range(n_imp):
        cand[b, cnt[b]:] = 0
        if cnt[b]:
            lab[b, rng.integers(0, cnt[b])] = 1
    return hist, hl, cand, cnt, lab


def _worker(rank, world, port, q):
    try:
        os.environ['MASTER_ADDR'] = '127.0.0.1'
        os.environ['MASTER_PORT'] = str(port)
        dist.init_process_group('gloo', rank=rank, world_size=world)
        Scorer = _scorer_class()
        m = _Model()
        # 300 news = 5 chunks of 64 (the last one partial); 44 = 1 chunk; 172 = 3 chunks
        for n_news in (300, 44, 172):
            fields = _corpus(n_news, seed=n_news)
            ref, sh = Scorer(m, *fields, chunk=64), Scorer(m, *fields, chunk=64, process_group=dist.group.WORLD)
            assert torch.equal(sh.encode_corpus(cuda_graph=False), ref.encode_corpus(cuda_graph=False)), n_news
            for n_imp in (150, 40, 64):
                hist, hl, cand, cnt, lab = _impressions(n_news, n_imp, seed=n_news + n_imp)
                s_sh = sh._impression_scores(hist, hl, cand, BATCH, cnt, lab)
                assert s_sh.shape == (n_imp, 6) and torch.equal(s_sh, ref._impression_scores(hist, hl, cand, BATCH))
                *m_sh, r_sh = sh.evaluate(hist, hl, cand, cnt, lab, batch=BATCH)
                *m_ref, r_ref = ref.evaluate(hist, hl, cand, cnt, lab, batch=BATCH)
                assert torch.equal(r_sh, r_ref) and m_sh == m_ref, (n_news, n_imp)
        # every rank raises, naming the fields, when one rank is called with other inputs; the ranks stay in step
        sh = Scorer(m, *_corpus(300, 300), chunk=64, process_group=dist.group.WORLD)
        sh.encode_corpus(cuda_graph=False)
        hist, hl, cand, cnt, lab = _impressions(300, 150, seed=3)
        n_imp = 150 - (rank == 1)
        with pytest.raises(RuntimeError, match=r'I: \[150, 149'):
            sh.evaluate(hist[:n_imp], hl[:n_imp], cand[:n_imp], cnt[:n_imp], lab[:n_imp], batch=BATCH)
        other = cand.copy()
        other[7, 0] += rank == 1
        with pytest.raises(RuntimeError, match='candidate_ids checksum') as err:
            sh.evaluate(hist, hl, other, cnt, lab, batch=BATCH)
        assert 'I:' not in str(err.value)
        with pytest.raises(RuntimeError, match='chunk'):
            Scorer(m, *_corpus(300, 300), chunk=64 + (rank == 1), process_group=dist.group.WORLD).encode_corpus(cuda_graph=False)
        assert sh.evaluate(hist, hl, cand, cnt, lab, batch=BATCH)[4].shape == (150, 6)
        q.put((rank, 'ok'))
    except BaseException as ex:
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        q.close()
        q.join_thread()
        os._exit(0)


@pytest.mark.parametrize('world', [2, 3, 4])
def test_sharded_scorer_host_logic_equals_plain_scorer(world):
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
