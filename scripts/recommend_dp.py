"""Data-parallel top-k recommendation: ``CorpusScorer.recommend(collective=True)`` over N GPUs, on the workloads of
scripts/recommend_bench.py: the synthetic 100 k-news corpus (seed 5, chunk 4096) and the config-2 model (seeded weights),
256 users x pools of 10 000 and 100 000 news with k = 10 and 100 at the default tile, one capped case (m = 2), and one user
x 100 000 news at T = 4096 (the case that splitting the users between ranks cannot help).

  python scripts/recommend_dp.py --gpus 1 2 4 8 [--group-of-one] [--reps 3] [--out FILE]

prints one JSON line per N (appended to FILE too) with, per workload: the median over --reps calls of the largest per-rank
call time (each call starts after a barrier; CUDA events), every rep's time, the all-gather of the rank lists plus the
final merge alone (the same events, on this rank's real list), the strong-scaling efficiency against N = 1 in the same run
(T1 / (N x TN)), and a SHA-256 of (ids, scores), which must be the same for every N; and the card name and power limit
read in the same run.  N = 1 is the plain scorer (no process group); with --group-of-one it is the collective path over an
NCCL group of one rank, timed alternately with the plain call, whose time and digest the line reports too."""
import argparse, hashlib, json, os, statistics, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from scoring_dp import _card, _free_port

# (users, pool, k, max_per_category, pool_tile); None tile = CorpusScorer.default_pool_tile(users)
WORKLOADS = [(256, 10000, 10, None, None), (256, 10000, 100, None, None), (256, 100000, 10, None, None),
             (256, 100000, 100, None, None), (256, 10000, 10, 2, None), (1, 100000, 10, None, 4096)]


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
                          syn.news_category, syn.news_subCategory, chunk=4096,
                          process_group=dist.group.WORLD if sharded else None)
        sc.encode_corpus()

        def barrier():
            if sharded:
                dist.barrier()
            torch.cuda.synchronize()

        def once(fn):
            """this rank's time of fn() in ms, started after a barrier"""
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1), out

        rows = []
        for B, P, k, mpc, tile in WORKLOADS:
            hist, hl, _ = syn.sample_behaviors(B, news_num=1, seed=1)
            hist, hl = torch.from_numpy(hist).to(dev), torch.from_numpy(hl).to(dev)
            pool = torch.from_numpy(np.random.default_rng(3).choice(a.news, P, replace=False)).to(dev)
            T = sc.default_pool_tile(B) if tile is None else tile
            call = lambda: sc.recommend(hist, hl, pool, k, pool_tile=T, max_per_category=mpc, collective=sharded)
            plain = lambda: sc.recommend(hist, hl, pool, k, pool_tile=T, max_per_category=mpc)
            fns = [call] + ([plain] if sharded and world == 1 else [])
            for fn in fns:
                fn()                                                  # warm-up: graph capture, NCCL channels
            ms = [[] for _ in fns]
            outs = [None] * len(fns)
            for r in range(a.reps):                                   # alternate the two paths of a group of one
                for i in (range(len(fns)) if r % 2 == 0 else reversed(range(len(fns)))):
                    t, outs[i] = once(fns[i])
                    ms[i].append(t)
            row = dict(users=B, pool=P, k=k, max_per_category=mpc, pool_tile=T, tiles=-(-P // T),
                       call_ms=statistics.median(ms[0]), call_ms_all=ms[0],
                       sha256=hashlib.sha256(outs[0][0].cpu().numpy().tobytes() + outs[0][1].cpu().numpy().tobytes()).hexdigest())
            if len(fns) == 2:
                row.update(plain_ms=statistics.median(ms[1]), plain_ms_all=ms[1],
                           plain_sha256=hashlib.sha256(outs[1][0].cpu().numpy().tobytes() +
                                                       outs[1][1].cpu().numpy().tobytes()).hexdigest())
            row['gather_merge_ms'] = None
            if sharded:
                # the all-gather of the rank lists and the final merge alone, on this rank's real list
                hid, hl_, pool_, k_, T_, m_, groups = sc._recommend_inputs(hist, hl, pool, k, True, T, mpc)
                first, end = contiguous_blocks(-(-P // T), world)[1][rank]
                mine = sc._recommend_tiles(hid, hl_, pool_, k_, T_, first, end, True, m_, groups, True)
                sc._gather_and_merge(mine, m_, groups)
                row['gather_merge_ms'] = statistics.median(once(lambda: sc._gather_and_merge(mine, m_, groups))[0]
                                                           for _ in range(max(a.reps, 5)))
            rows.append(row)
        name, watts = _card(rank)
        q.put((rank, dict(rows=rows, card=name, power_limit_w=watts)))
    except BaseException as ex:
        import traceback
        q.put((rank, 'FAILED: %s\n%s' % (ex, traceback.format_exc())))
    finally:
        sys.stdout.flush()
        q.close()
        q.join_thread()
        os._exit(0)                                                   # no destroy_process_group(): the process ends here


def run(world, a):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, a)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=3600) for _ in range(world))
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.kill()
    for r in range(world):
        if not isinstance(res[r], dict):
            raise RuntimeError('N=%d rank %d: %s' % (world, r, res[r]))
    ranks = [res[r]['rows'] for r in range(world)]
    workloads = []
    for i, row in enumerate(ranks[0]):
        assert all(x[i]['sha256'] == row['sha256'] for x in ranks), ('ranks disagree', i)
        out = dict(row)
        for key in ('call_ms', 'plain_ms', 'gather_merge_ms'):       # the slowest rank
            if out.get(key) is not None:
                out[key] = max(x[i][key] for x in ranks)
        out['call_ms_all'] = [max(x[i]['call_ms_all'][j] for x in ranks) for j in range(len(row['call_ms_all']))]
        out['pairs_per_sec'] = row['users'] * row['pool'] / (out['call_ms'] * 1e-3)
        workloads.append(out)
    return {'gpus': world, 'sharded': world > 1 or a.group_of_one, 'corpus_news': a.news, 'reps': a.reps,
            'workloads': workloads, 'card': sorted({res[r]['card'] for r in range(world)}),
            'power_limit_w': sorted({res[r]['power_limit_w'] for r in range(world)}, key=str)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, nargs='+', default=[1])
    ap.add_argument('--news', type=int, default=100000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--group-of-one', action='store_true',
                    help='at N = 1, run the collective path over an NCCL group of one rank, alternated with the plain call')
    ap.add_argument('--out', help='also append the JSON lines to this file')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('recommend_dp.py needs CUDA devices')
    if max(a.gpus) > torch.cuda.device_count():
        sys.exit('--gpus %s: only %d CUDA devices' % (a.gpus, torch.cuda.device_count()))
    base = None
    for world in a.gpus:
        line = run(world, a)
        line['time'] = time.strftime('%Y-%m-%dT%H:%M:%S')
        if world == 1:
            base = line
        if base is not None:
            for w, b in zip(line['workloads'], base['workloads']):
                w['efficiency'] = b['call_ms'] / (world * w['call_ms'])
                w['same_results_as_1_gpu'] = w['sha256'] == b['sha256']
        print(json.dumps(line), flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
