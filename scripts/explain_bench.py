"""What explaining a click score costs: ``CorpusScorer.explain`` against ``score`` on the workload of
``scoring_dp.py --factored`` (bench.py's synthetic 100 k-news corpus, seed 5, chunk 4096; 16 384 impressions at batch
256), once with 37 candidates each and once on the ragged set (seeded long-tailed counts, mean about 37, padded to 300 with
-1 ids).

  python scripts/explain_bench.py [--reps 3] [--out FILE]

For each set, every batch is timed through four calls, alternated pair by pair in the same run (the median over --reps
passes of the whole set):
  * explain(exact=False) against score(exact=False) of the same entries: its argument checks, then the packed factored
    tail of the valid entries, which score() runs with all n entries valid and evaluate(exact=False) with the counts;
  * explain(exact=True) against score() (what evaluate(exact=True) scores: every padded entry, padding as news 0).
Then explain(exact=False / True) of a recommend(k=10, exact=False) result for 256 users over the whole corpus, fill
entries included (the recommend call itself is not timed).  Each line records the times, their ratios, whether the
explained scores equal the scores bit for bit, the largest |sum_c cluster_score - score| / sum_c |cluster_score|, SHA-256
digests of the outputs, and the card name and power limit read in the same run.  One JSON line per measurement is
printed and, with --out, appended to FILE."""
import argparse, hashlib, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from scoring_dp import _card, ragged_counts


def _digest(tensors):
    h = hashlib.sha256()
    for t in tensors:
        if t is not None:
            h.update(t.contiguous().cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def _alternated(fns, reps):
    """median ms of each of fns (name -> callable), called in turn, reps times each"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for fn in fns.values():                                          # warm-up: graph captures
        fn()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    return {k: sorted(v)[len(v) // 2] for k, v in ms.items()}, ms


def _checks(explanations, scores):
    """explained scores equal to the scores bit for bit; the largest |sum_c cluster_score - score| / sum_c |cluster_score|"""
    same, worst = True, 0.0
    for e, s in zip(explanations, scores):
        same &= torch.equal(e.scores.contiguous().view(torch.int32), s.contiguous().view(torch.int32))
        if e.cluster_score is not None:
            gap = (e.cluster_score.sum(2) - e.scores).abs() / e.cluster_score.abs().sum(2).clamp(min=1e-30)
            worst = max(worst, gap.max().item())
    return bool(same), worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--news', type=int, default=100000)
    ap.add_argument('--impressions', type=int, default=16384)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--users', type=int, default=256)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', help='also append the JSON lines to this file')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('explain_bench.py needs a CUDA device')
    import nnr_b200
    from nnr_b200.scoring import CorpusScorer
    from nnr_b200.synthetic import SyntheticMIND
    from bench import make_config

    class Args:
        vocab, dropout = 40000, 0.2
    dev = torch.device('cuda', 0)
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
    card, watts = _card(0)
    lines = []

    def emit(line):
        line.update(card=card, power_limit_w=watts, reps=a.reps, time=time.strftime('%Y-%m-%dT%H:%M:%S'))
        print(json.dumps(line), flush=True)
        lines.append(line)

    B = a.batch
    for ragged in (False, True):
        n_max = 300 if ragged else 37
        hist, hl, cand = syn.sample_behaviors(a.impressions, news_num=n_max, seed=1)
        cnt = ragged_counts(a.impressions, n_max) if ragged else np.full(a.impressions, n_max)
        cand = np.where(np.arange(n_max)[None, :] < cnt[:, None], cand, -1)
        hist, hl, cand, cnt = (torch.from_numpy(x).to(dev) for x in (hist, hl, cand, cnt))
        exact_cand = torch.where(cand >= 0, cand, 0)               # the exact path reads the padding entries too
        span = range(0, a.impressions, B)

        def factored_score(s):
            """score(exact=False) of a batch, given its counts: the same checks, then the same packed scoring"""
            cid, c = sc._packed_inputs('score', cand[s:s + B], cnt[s:s + B])
            return sc._score_packed(hist[s:s + B], hl[s:s + B], cid, c, True)

        calls = {
            'factored_score': lambda: [factored_score(s) for s in span],
            'factored_explain': lambda: [sc.explain(hist[s:s + B], hl[s:s + B], cand[s:s + B], cnt[s:s + B]) for s in span],
            'exact_score': lambda: [sc.score(hist[s:s + B], hl[s:s + B], exact_cand[s:s + B]) for s in span],
            'exact_explain': lambda: [sc.explain(hist[s:s + B], hl[s:s + B], cand[s:s + B], cnt[s:s + B], exact=True)
                                      for s in span],
        }
        med, ms = _alternated(calls, a.reps)
        line = {'workload': 'ragged' if ragged else '37 candidates', 'corpus_news': a.news, 'impressions': a.impressions,
                'n_max': n_max, 'batch': B, 'pairs': int(cnt.sum())}
        for path in ('factored', 'exact'):
            scores, expl = calls[path + '_score'](), calls[path + '_explain']()
            if path == 'exact':                                    # explain() zeroes the entries past the counts
                valid = torch.arange(n_max, device=dev)[None, :] < cnt[:, None]
                scores = [torch.where(valid[s:s + B], x, 0.0) for s, x in zip(span, scores)]
            same, gap = _checks(expl, scores)
            line.update({path + '_score_ms': med[path + '_score'], path + '_explain_ms': med[path + '_explain'],
                         path + '_score_ms_all': ms[path + '_score'], path + '_explain_ms_all': ms[path + '_explain'],
                         path + '_explain_over_score': med[path + '_explain'] / med[path + '_score'],
                         path + '_scores_equal_score': same, path + '_max_cluster_sum_gap': gap,
                         path + '_digests': {f: _digest([getattr(e, f) for e in expl]) for f in expl[0]._fields}})
        emit(line)

    hist, hl, _ = syn.sample_behaviors(a.users, news_num=1, seed=7)
    hist, hl = torch.from_numpy(hist).to(dev), torch.from_numpy(hl).to(dev)
    ids, rs = sc.recommend(hist, hl, torch.arange(a.news), 10, exact=False)
    cnt = (ids >= 0).sum(1)
    calls = {'factored': lambda: sc.explain(hist, hl, ids, cnt), 'exact': lambda: sc.explain(hist, hl, ids, cnt, exact=True)}
    med, ms = _alternated(calls, a.reps)
    line = {'workload': 'recommend(k=10, exact=False) result', 'corpus_news': a.news, 'pool': a.news, 'users': a.users}
    for path in ('factored', 'exact'):
        e = calls[path]()
        filled = ids >= 0
        line.update({path + '_explain_ms': med[path], path + '_explain_ms_all': ms[path],
                     path + '_max_rel_score_deviation': ((e.scores - rs).abs()[filled].max() / rs[filled].abs().max()).item(),
                     path + '_digests': {f: _digest([getattr(e, f)]) for f in e._fields}})
    emit(line)
    if a.out:
        with open(a.out, 'a') as f:
            for line in lines:
                f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
