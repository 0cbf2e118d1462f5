"""Top-k recommendation over a candidate pool: ``CorpusScorer.recommend`` against today's workaround (``score()`` per pool
tile, the [B, T] rows copied to the host, concatenated and ``torch.topk``-ed there), on the inputs of bench.py's
``extra.scoring``: the synthetic 100 k-news corpus (seed 5, chunk 4096) and the config-2 model (seeded weights).

  python scripts/recommend_bench.py [--users 256] [--pools 1000 10000 100000] [--ks 10 100] [--out FILE]
                                    [--max-per-category M [M ...] | --factored]

prints one JSON line per (P, k) (appended to FILE too): ms per call and (user, candidate) pairs/s of both paths on the same
users and pool (median over --reps calls, host clock around calls that end in a device synchronise, after one warm-up
call that captures the graphs); the share of recommend's time spent in nnr_topk_merge (CUDA events around every merge,
in a separate pass); peak torch.cuda.max_memory_allocated of each path, over what was allocated before the call and
absolute, and the memory the warm-up call left allocated (the captured graphs' pools, held while the scorer lives); whether
the two paths return the same top-k scores (recommend without exclusion; checked for P <= --check-max); the card name
and power limit read in the same run.

With --factored, one line per (P, k) instead: recommend(exact=False) (the factored cluster tail, its default tile) against
recommend(exact=True) on the same users and pool, the two alternated call by call (--reps each, medians and every time);
the speed ratio; the largest deviation of the returned scores from the exact scores of the same ids (score() of the
returned ids, max |factored - exact| / max |exact| over the [B, k] entries); the mean overlap of the two id lists (|common
ids| / k per user); the card name and power limit.

With --max-per-category, one line per (P, k, m) instead: recommend(max_per_category=m) against the uncapped call on the
same users and pool, the two alternated call by call (--reps each, medians and every time); the merge's share of each
call (CUDA events around every nnr_topk_merge / nnr_topk_merge_capped, in a separate pass); the largest number of one
category in a user's list, averaged over the users, for both; SHA-256 digests of both outputs (ids and scores); the card
name and power limit."""
import argparse, hashlib, json, os, statistics, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch


def card():
    """(name, power limit in W) of the current device"""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader,nounits',
                              '-i', str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout
        name, watts = [x.strip() for x in out.strip().splitlines()[0].split(',')]
        return name, float(watts)
    except Exception:
        return torch.cuda.get_device_name(), None


def timed(fn, reps):
    """median host time in ms of fn() followed by a device synchronise, and the last result"""
    ts, out = [], None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def merge_time(fn, ops, name):
    """(ms summed over CUDA events around every ops.<name> call during one fn(), that over fn()'s host time)"""
    spans, merge = [], getattr(ops, name)

    def merge_timed(*args, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        merge(*args, **kw)
        e1.record()
        spans.append((e0, e1))
    setattr(ops, name, merge_timed)
    try:
        total_ms, _ = timed(fn, 1)
    finally:
        setattr(ops, name, merge)
    ms = sum(e0.elapsed_time(e1) for e0, e1 in spans)
    return ms, ms / total_ms


def digest(ids, scores):
    return hashlib.sha256(ids.cpu().numpy().tobytes() + scores.cpu().numpy().tobytes()).hexdigest()


def crowding(ids, cat):
    """the largest number of news of one category in a user's list, averaged over the users"""
    c = cat[ids.clamp(min=0)].long()
    c[ids < 0] = -1
    counts = torch.stack([(c == g).sum(1) for g in range(int(cat.max()) + 1)], 1)
    return float(counts.max(1)[0].float().mean())


def capped_lines(a, sc, ops, hist, hl, pool, P, T, name, watts):
    """--max-per-category: one line per (k, m), capped against uncapped calls alternated in the same run"""
    B = hist.shape[0]
    for k in a.ks:
        unc = lambda: sc.recommend(hist, hl, pool, k)
        unc()                                                         # warm-up: graph capture, workspaces
        unc_out = unc()
        unc_merge_ms, unc_share = merge_time(unc, ops, 'topk_merge')
        for m in a.max_per_category:
            cap = lambda: sc.recommend(hist, hl, pool, k, max_per_category=m)
            cap_out = cap()                                           # warm-up
            t_unc, t_cap = [], []
            for r in range(a.reps):                                   # alternate, and alternate which goes first
                for fn, ts in ((unc, t_unc), (cap, t_cap))[::1 if r % 2 == 0 else -1]:
                    ts.append(timed(fn, 1)[0])
            cap_merge_ms, cap_share = merge_time(cap, ops, 'topk_merge_capped')
            u, c = statistics.median(t_unc), statistics.median(t_cap)
            line = dict(users=B, pool=P, k=k, max_per_category=m, pool_tile=T, tiles=-(-P // T), corpus_news=a.news,
                        history=hist.shape[1], uncapped_ms=u, capped_ms=c, capped_over_uncapped=c / u,
                        uncapped_ms_all=t_unc, capped_ms_all=t_cap, capped_pairs_per_sec=B * P / (c * 1e-3),
                        uncapped_merge_ms=unc_merge_ms, uncapped_merge_share=unc_share, capped_merge_ms=cap_merge_ms,
                        capped_merge_share=cap_share, uncapped_max_per_category_mean=crowding(unc_out[0], sc.cat),
                        capped_max_per_category_mean=crowding(cap_out[0], sc.cat),
                        uncapped_digest=digest(*unc_out), capped_digest=digest(*cap_out),
                        card=name, power_limit_w=watts, time=time.strftime('%Y-%m-%dT%H:%M:%S'))
            print(json.dumps(line), flush=True)
            if a.out:
                with open(a.out, 'a') as f:
                    f.write(json.dumps(line) + '\n')


def emit(a, line):
    print(json.dumps(line), flush=True)
    if a.out:
        with open(a.out, 'a') as f:
            f.write(json.dumps(line) + '\n')


def factored_lines(a, sc, hist, hl, pool, P, name, watts):
    """--factored: one line per k, recommend(exact=False) against recommend(exact=True) alternated in the same run"""
    B = hist.shape[0]
    for k in a.ks:
        exact = lambda: sc.recommend(hist, hl, pool, k)
        fact = lambda: sc.recommend(hist, hl, pool, k, exact=False)
        ex_out, fa_out = exact(), fact()                              # warm-up: graph capture, workspaces
        t_ex, t_fa = [], []
        for r in range(a.reps):                                       # alternate, and alternate which goes first
            for fn, ts in ((exact, t_ex), (fact, t_fa))[::1 if r % 2 == 0 else -1]:
                ts.append(timed(fn, 1)[0])
        ids, scores = fa_out
        real = ids >= 0
        ref = sc.score(hist, hl, ids.clamp(min=0), cuda_graph=False)  # exact scores of the returned ids
        dev = float(((scores - ref).abs() * real).max() / (ref.abs() * real).max())
        overlap = float(np.mean([len(set(f.tolist()) & set(e.tolist()) - {-1}) / min(k, P)
                                 for f, e in zip(ids.cpu(), ex_out[0].cpu())]))
        e, f = statistics.median(t_ex), statistics.median(t_fa)
        emit(a, dict(users=B, pool=P, k=k, factored_pool_tile=min(P, 4096), exact_pool_tile=sc.default_pool_tile(B),
                     corpus_news=a.news, history=hist.shape[1], exact_ms=e, factored_ms=f, speed_ratio=e / f,
                     exact_ms_all=t_ex, factored_ms_all=t_fa, factored_pairs_per_sec=B * P / (f * 1e-3),
                     max_rel_score_deviation=dev, mean_id_overlap=overlap, card=name, power_limit_w=watts,
                     time=time.strftime('%Y-%m-%dT%H:%M:%S')))


def peak_mb(fn):
    """(peak over what was allocated before the call, absolute peak) of torch.cuda.max_memory_allocated during fn(), MiB"""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    return (peak - base) / 2 ** 20, peak / 2 ** 20


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--news', type=int, default=100000)
    ap.add_argument('--users', type=int, default=256)
    ap.add_argument('--pools', type=int, nargs='+', default=[1000, 10000, 100000])
    ap.add_argument('--ks', type=int, nargs='+', default=[10, 100])
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--check-max', type=int, default=10000, help='largest P whose top-k scores are compared between the paths')
    ap.add_argument('--out', default=None)
    ap.add_argument('--max-per-category', type=int, nargs='+', default=None,
                    help='time recommend(max_per_category=m) against the uncapped call, for each m')
    ap.add_argument('--factored', action='store_true', help='time recommend(exact=False) against recommend(exact=True)')
    a = ap.parse_args()
    import nnr_b200
    from nnr_b200 import ops
    from nnr_b200.scoring import CorpusScorer
    from nnr_b200.synthetic import SyntheticMIND
    from bench import make_config

    class Args:
        vocab, dropout = 40000, 0.2
    dev = torch.device('cuda')
    cfg = make_config(Args)
    syn = SyntheticMIND(news_num=a.news, vocabulary_size=40000, lengths='mind', seed=5)
    cfg.pretrained_word_embedding = syn.word_table()
    torch.manual_seed(1234)
    m = nnr_b200.Model(cfg)
    m.initialize()
    m.to(dev).eval()
    sc = CorpusScorer(m, syn.news_title_text, syn.news_title_mask, syn.news_abstract_text, syn.news_abstract_mask,
                      syn.news_category, syn.news_subCategory, chunk=4096)
    sc.encode_corpus()
    hist, hl, _ = syn.sample_behaviors(a.users, news_num=1, seed=1)
    hist, hl = torch.from_numpy(hist).to(dev), torch.from_numpy(hl).to(dev)
    B = a.users
    T = sc.default_pool_tile(B)
    name, watts = card()
    for P in a.pools:
        pool = torch.from_numpy(np.random.default_rng(3).choice(a.news, P, replace=False)).to(dev)
        if a.max_per_category:
            capped_lines(a, sc, ops, hist, hl, pool, P, T, name, watts)
            continue
        if a.factored:
            factored_lines(a, sc, hist, hl, pool, P, name, watts)
            continue
        for k in a.ks:
            rec = lambda: sc.recommend(hist, hl, pool, k)

            def workaround():
                rows = [sc.score(hist, hl, pool[i:i + T].expand(B, -1)).cpu() for i in range(0, P, T)]
                s, j = torch.topk(torch.cat(rows, 1), min(k, P), dim=1)
                return pool.cpu()[j], s

            torch.cuda.synchronize()
            before = torch.cuda.memory_allocated()
            rec()                                                     # warm-up: graph capture, workspaces
            torch.cuda.synchronize()
            retained_mb = (torch.cuda.memory_allocated() - before) / 2 ** 20   # captured graph pools (first case of a tile)
            rec_ms, _ = timed(rec, a.reps)
            rec_mb = peak_mb(rec)
            topk_ms, topk_share = merge_time(rec, ops, 'topk_merge')  # top-k pass: CUDA events around every merge
            sc.score(hist, hl, pool[:T].expand(B, -1))                # warm-up of score()'s graph for a full tile
            wa_ms, (_, wa_scores) = timed(workaround, a.reps)
            wa_mb = peak_mb(workaround)
            same = None
            if P <= a.check_max:
                ids, scores = sc.recommend(hist, hl, pool, k, exclude_history=False)
                same = bool(torch.equal(scores[:, :min(k, P)].cpu(), wa_scores))
            line = dict(users=B, pool=P, k=k, pool_tile=T, tiles=-(-P // T), corpus_news=a.news, history=hist.shape[1],
                        recommend_ms=rec_ms, recommend_pairs_per_sec=B * P / (rec_ms * 1e-3),
                        topk_merge_ms=topk_ms, topk_share=topk_share, recommend_peak_mb=rec_mb[0],
                        recommend_peak_abs_mb=rec_mb[1], recommend_warmup_retained_mb=retained_mb,
                        tiled_score_topk_ms=wa_ms, tiled_score_topk_pairs_per_sec=B * P / (wa_ms * 1e-3),
                        tiled_score_topk_peak_mb=wa_mb[0], tiled_score_topk_peak_abs_mb=wa_mb[1], speed_ratio=wa_ms / rec_ms, same_topk_scores=same,
                        card=name, power_limit_w=watts, time=time.strftime('%Y-%m-%dT%H:%M:%S'))
            print(json.dumps(line), flush=True)
            if a.out:
                with open(a.out, 'a') as f:
                    f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
