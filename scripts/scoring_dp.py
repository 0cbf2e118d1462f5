"""Data-parallel dev scoring: ``CorpusScorer`` with a process group over N GPUs, on the inputs of bench.py's
``extra.scoring`` (a synthetic 100 k-news corpus, seed 5, chunk 4096) plus 16 384 impressions x 37 candidates scored at
batch 256 with on-device ranking and metrics.

  python scripts/scoring_dp.py --gpus 1 2 4 8 [--out FILE]

prints one JSON line per N (appended to FILE too): encode ms and the all-gather of the encoded corpus alone, evaluate ms
(scores + ranking + metrics) and impressions/s, the score all-gather inside it alone, the strong-scaling efficiency against
N = 1 (T1 / (N x TN)) when N = 1 is in the same run, the card name and power limit read in the same run, and a digest of
the cache and the four metrics, which must be the same for every N.  N = 1 is the plain scorer (no process group),
or with --group-of-one the sharded path over an NCCL group of one rank.
Times are the median over --reps calls of the largest per-rank time (each call starts after a barrier).

  python scripts/scoring_dp.py --gpus 1 --factored [--ragged] [--out FILE]

--factored times evaluate(exact=True) and evaluate(exact=False) (the factored cluster tail, packed by candidate count)
alternated call by call in the same run, and adds for each path: evaluate ms, impressions/s, pairs/s (the sum of the
candidate counts over the time), the peak memory allocated during the first call (graph captures and their memory pools
included), and the speedup; the largest deviation of
the valid exact=False scores from the exact ones (max |F - S| / max |S|); both paths' metrics and their differences; the
fraction of impressions whose ranks differ.  --ragged draws seeded long-tailed candidate counts (lognormal, mean about 37,
clipped to [2, 300]) over impressions padded to n_max = 300 with -1 ids, MIND-like (the 37-candidate workload pads
nothing), and records the count distribution."""
import argparse, hashlib, json, os, socket, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _card(index):
    """(name, power limit in W) of a device, read through NVML"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        name = pynvml.nvmlDeviceGetName(h)
        return (name.decode() if isinstance(name, bytes) else name), pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception:
        return torch.cuda.get_device_name(index), None


def _worker(rank, world, port, q, a):
    try:
        import numpy as np
        import torch.distributed as dist
        torch.cuda.set_device(rank)
        dev = torch.device('cuda', rank)
        sharded = world > 1 or a.group_of_one
        if sharded:
            os.environ['MASTER_ADDR'] = '127.0.0.1'
            os.environ['MASTER_PORT'] = str(port)
            dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
        import nnr_b200
        from nnr_b200.scoring import CorpusScorer, contiguous_blocks
        from nnr_b200.synthetic import SyntheticMIND
        from bench import make_config

        class Args:
            vocab, dropout = 40000, 0.2
        cfg = make_config(Args)
        syn = SyntheticMIND(news_num=a.news, vocabulary_size=40000, lengths='mind', seed=5)
        cfg.pretrained_word_embedding = syn.word_table()
        torch.manual_seed(1234)                                       # the same weights on every rank
        m = nnr_b200.Model(cfg)
        m.initialize()
        m.to(dev).eval()
        sc = CorpusScorer(m, syn.news_title_text, syn.news_title_mask, syn.news_abstract_text, syn.news_abstract_mask,
                          syn.news_category, syn.news_subCategory, chunk=a.chunk,
                          process_group=dist.group.WORLD if sharded else None)
        hist, hl, cand = syn.sample_behaviors(a.impressions, news_num=a.candidates, seed=1)
        rng = np.random.default_rng(2)
        cnt = np.full(a.impressions, a.candidates)
        if a.ragged:
            cnt = ragged_counts(a.impressions, a.candidates)
            cand = np.where(np.arange(a.candidates)[None, :] < cnt[:, None], cand, -1)
        lab = np.zeros(cand.shape, dtype=np.int64)
        lab[np.arange(a.impressions), rng.integers(0, cnt if a.ragged else a.candidates, size=a.impressions)] = 1
        hist, hl, cand, cnt, lab = (torch.from_numpy(x).to(dev) for x in (hist, hl, cand, cnt, lab))

        def barrier():
            if sharded:
                dist.barrier()
            torch.cuda.synchronize()

        def timed(fn):
            """median over reps of this rank's time of fn(), each call started after a barrier"""
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            fn()                                                      # warm-up: graph captures, NCCL channels
            ms = []
            for _ in range(a.reps):
                barrier()
                e0.record()
                out = fn()
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
            return sorted(ms)[len(ms) // 2], out

        D = m.news_encoder.news_embedding_dim
        enc_ms, cache = timed(sc.encode_corpus)
        if a.factored:
            q.put((rank, factored(sc, hist, hl, cand, cnt, lab, a, barrier) | dict(card=_card(rank)[0],
                                                                                   power_limit_w=_card(rank)[1])))
            return
        eval_ms, res = timed(lambda: sc.evaluate(hist, hl, cand, cnt, lab, batch=a.batch))
        res_digest = hashlib.sha256(cache.cpu().numpy().tobytes()).hexdigest()[:16]
        rank_digest = hashlib.sha256(res[4].cpu().numpy().tobytes()).hexdigest()[:16]
        ag_ms = ag_eval_ms = None
        if sharded:
            # the two all-gathers alone, at the sizes the calls above use
            k, _ = contiguous_blocks(-(-a.news // a.chunk), world)
            send, recv = torch.zeros(k * a.chunk, D, device=dev), torch.empty(world * k * a.chunk, D, device=dev)
            ag_ms, _ = timed(lambda: dist.all_gather_into_tensor(recv, send))
            kb, _ = contiguous_blocks(-(-a.impressions // a.batch), world)
            send, recv = torch.zeros(kb * a.batch, a.candidates, device=dev), torch.empty(world * kb * a.batch, a.candidates, device=dev)
            ag_eval_ms, _ = timed(lambda: dist.all_gather_into_tensor(recv, send))
        name, watts = _card(rank)
        q.put((rank, dict(encode_ms=enc_ms, allgather_ms=ag_ms, evaluate_ms=eval_ms, score_allgather_ms=ag_eval_ms,
                          metrics=list(res[:4]), cache_sha256=res_digest, ranks_sha256=rank_digest, card=name, power_limit_w=watts)))
    except BaseException as ex:
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        sys.stdout.flush()
        q.close()
        q.join_thread()
        os._exit(0)                                                   # no destroy_process_group(): the process ends here


def ragged_counts(impressions, n_max):
    """seeded long-tailed candidate counts: lognormal with mean about 37, clipped to [2, n_max] (one positive and one
    negative at least)"""
    import numpy as np
    rng = np.random.default_rng(3)
    return np.clip(np.round(rng.lognormal(np.log(37.0) - 0.5 * 0.9 ** 2, 0.9, impressions)), 2, n_max).astype(np.int64)


def factored(sc, hist, hl, cand, cnt, lab, a, barrier):
    """evaluate(exact=True) and evaluate(exact=False) alternated call by call: times, peak memory, score deviation,
    metrics and rank agreement"""
    exact_cand = torch.where(cand >= 0, cand, 0)                  # the exact path reads the padding entries too
    ev = {True: lambda: sc.evaluate(hist, hl, exact_cand, cnt, lab, batch=a.batch),
          False: lambda: sc.evaluate(hist, hl, cand, cnt, lab, batch=a.batch, exact=False)}
    res, ms, peak = {}, {True: [], False: []}, {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for exact in (True, False):
        # the first call captures the graphs: its peak includes their memory pools, which later replays reuse
        barrier()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        res[exact] = ev[exact]()
        torch.cuda.synchronize()
        peak[exact] = torch.cuda.max_memory_allocated() - base
    for _ in range(a.reps):
        for exact in (True, False):
            barrier()
            e0.record()
            ev[exact]()
            e1.record()
            torch.cuda.synchronize()
            ms[exact].append(e0.elapsed_time(e1))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    S = sc._impression_scores(hist, hl, exact_cand, a.batch)
    F = sc._impression_scores(hist, hl, cand, a.batch, cnt, lab, exact=False)
    valid = torch.arange(cand.shape[1], device=S.device)[None, :] < cnt[:, None]
    dev = ((F - S).abs()[valid].max() / S[valid].abs().max()).item()
    pairs = int(cnt.sum())
    out = {}
    for exact, name in ((True, 'exact'), (False, 'factored')):
        out.update({name + '_evaluate_ms': med[exact], name + '_evaluate_ms_all': ms[exact],
                    name + '_impressions_per_sec': len(cnt) / (med[exact] * 1e-3),
                    name + '_pairs_per_sec': pairs / (med[exact] * 1e-3), name + '_peak_allocated_bytes': peak[exact],
                    name + '_metrics': list(res[exact][:4])})
    out.update(speedup=med[True] / med[False], pairs=pairs, max_rel_score_deviation=dev,
               metric_differences=[f - e for f, e in zip(res[False][:4], res[True][:4])],
               ranks_differ_fraction=(res[True][4] != res[False][4]).any(1).double().mean().item())
    return out


def run(world, a):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, a)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=1200) for _ in range(world))
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    for r in range(world):
        if not isinstance(res[r], dict):
            raise RuntimeError('N=%d rank %d: %s' % (world, r, res[r]))
    rows = [res[r] for r in range(world)]
    if a.factored:
        import numpy as np
        line = {'gpus': world, 'corpus_news': a.news, 'impressions': a.impressions, 'n_max': a.candidates,
                'batch': a.batch, 'ragged': a.ragged, 'reps': a.reps, **rows[0], 'card': [rows[0]['card']],
                'power_limit_w': [rows[0]['power_limit_w']]}
        if a.ragged:
            c = ragged_counts(a.impressions, a.candidates)
            line['counts'] = {'mean': float(c.mean()), 'median': float(np.median(c)), 'p90': float(np.percentile(c, 90)),
                              'p99': float(np.percentile(c, 99)), 'min': int(c.min()), 'max': int(c.max()),
                              'padded_over_valid': a.candidates * len(c) / float(c.sum()), 'seed': 3}
        return line
    for key in ('metrics', 'cache_sha256', 'ranks_sha256'):
        assert all(x[key] == rows[0][key] for x in rows), ('ranks disagree', key, [x[key] for x in rows])
    worst = lambda key: None if rows[0][key] is None else max(x[key] for x in rows)
    return {'gpus': world, 'sharded': world > 1 or a.group_of_one, 'corpus_news': a.news, 'chunk': a.chunk, 'impressions': a.impressions,
            'candidates_per_impression': a.candidates, 'batch': a.batch, 'encode_ms': worst('encode_ms'),
            'allgather_ms': worst('allgather_ms'), 'evaluate_ms': worst('evaluate_ms'),
            'score_allgather_ms': worst('score_allgather_ms'),
            'impressions_per_sec': a.impressions / (worst('evaluate_ms') * 1e-3), 'news_per_sec': a.news / (worst('encode_ms') * 1e-3),
            'metrics': rows[0]['metrics'], 'cache_sha256': rows[0]['cache_sha256'], 'ranks_sha256': rows[0]['ranks_sha256'],
            'card': sorted({x['card'] for x in rows}), 'power_limit_w': sorted({x['power_limit_w'] for x in rows}, key=str)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, nargs='+', default=[1])
    ap.add_argument('--news', type=int, default=100000)
    ap.add_argument('--impressions', type=int, default=16384)
    ap.add_argument('--candidates', type=int, default=37)
    ap.add_argument('--chunk', type=int, default=4096)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--group-of-one', action='store_true',
                    help='at N = 1, score over an NCCL group of one rank (the sharded code path) instead of the plain scorer')
    ap.add_argument('--factored', action='store_true',
                    help='time evaluate(exact=True) against evaluate(exact=False), alternated in the same run (one GPU)')
    ap.add_argument('--ragged', action='store_true',
                    help='seeded long-tailed candidate counts (mean about 37) padded to --candidates (default 300)')
    ap.add_argument('--out', help='also append the JSON lines to this file')
    a = ap.parse_args()
    if a.ragged and not a.factored:
        sys.exit('--ragged needs --factored')
    if a.factored and a.gpus != [1]:
        sys.exit('--factored runs on one GPU: --gpus 1')
    if a.ragged and '--candidates' not in sys.argv:
        a.candidates = 300
    if not torch.cuda.is_available():
        sys.exit('scoring_dp.py needs CUDA devices')
    if max(a.gpus) > torch.cuda.device_count():
        sys.exit('--gpus %s: only %d CUDA devices' % (a.gpus, torch.cuda.device_count()))
    base = None
    for world in a.gpus:
        line = run(world, a)
        line['time'] = time.strftime('%Y-%m-%dT%H:%M:%S')
        if world == 1 and not a.factored:
            base = line
        if base is not None:
            line['encode_efficiency'] = base['encode_ms'] / (world * line['encode_ms'])
            line['evaluate_efficiency'] = base['evaluate_ms'] / (world * line['evaluate_ms'])
            line['same_results_as_1_gpu'] = (line['cache_sha256'], line['ranks_sha256'], line['metrics']) == \
                (base['cache_sha256'], base['ranks_sha256'], base['metrics'])
        print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
