"""CPU tests that PIN the restated test infrastructure against the reference itself, executed (skipped where
no checkout of the original NNR project is found at NNR_REFERENCE_ROOT):

  * oracle/graph.py           against the literal source lines MIND_corpus.py:178-213 run under stub variables
                              (MIND_corpus.py cannot be imported: it needs nltk / torchtext at module level)
  * oracle/metrics.py         against evaluate.py imported live (ranking lines of util.py:52-62 executed from source)
  * the gcn_layer_norm / no_gcn_residual flags of the oracle against the live reference model

Committed goldens made by these same executions (tests/golden/graph_flags.npz, metrics.npz, via
tests/golden/make_golden.py) carry the pin to machines without the reference.
"""
import importlib.util
import io
import json
import os
import textwrap
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import graph as G
from oracle import metrics as OM
from oracle import nnr_oracle as O
from oracle import reference_import as R
from tests.util import GOLDEN_DIR

needs_reference = pytest.mark.skipif(not R.available(), reason='needs a checkout of the original NNR project at NNR_REFERENCE_ROOT; '
                                     'the *_committed_reference_vectors tests check against its stored outputs')

FLAG_SETS = [dict(no_self_connection=False, no_adjacent_normalization=False, gcn_normalization_type='symmetric'),
             dict(no_self_connection=False, no_adjacent_normalization=False, gcn_normalization_type='asymmetric'),
             dict(no_self_connection=False, no_adjacent_normalization=True, gcn_normalization_type='symmetric'),
             dict(no_self_connection=True, no_adjacent_normalization=True, gcn_normalization_type='symmetric')]


def reference_graph_source():
    """MIND_corpus.py:179-213 (the body of the per-behaviour loop after the line is split), dedented"""
    with open(os.path.join(R.REFERENCE_ROOT, 'MIND_corpus.py')) as f:
        lines = f.readlines()
    body = ''.join(lines[178:213])
    assert 'config.no_self_connection' in lines[178] and 'D_inv_sqrt), history_graph), D_inv_sqrt' not in lines[178]
    assert 'np.matmul(np.matmul(D_inv_sqrt, history_graph), D_inv_sqrt)' in lines[212]
    return textwrap.dedent(body)


def run_reference_graph(code, cats, H, C, flags):
    """execute the reference lines for one behaviour whose (already truncated) history has categories `cats`"""
    ids = ['N%d' % i for i in range(len(cats))]
    env = dict(np=np, config=SimpleNamespace(max_history_num=H, **flags), history=' '.join(ids),
               news_category_dict={n: int(c) for n, c in zip(ids, cats)}, category_num=C, graph_size=H + C)
    exec(code, env)
    return env['history_graph'], env['history_category_mask'], env['history_category_indices']


def graph_cases(seed=0, n=40, H=12, C=5):
    rng = np.random.default_rng(seed)
    out = [[], [0], [1, 1, 1], list(rng.integers(0, C, size=H))]
    for _ in range(n):
        out.append(list(rng.integers(0, C, size=int(rng.integers(0, H + 1)))))
    return out, H, C


@needs_reference
@pytest.mark.parametrize('flags', FLAG_SETS, ids=lambda f: '%s-%s-%s' % (f['no_self_connection'], f['no_adjacent_normalization'], f['gcn_normalization_type']))
def test_graph_restatement_equals_executed_reference_source(flags):
    code = compile(reference_graph_source(), 'MIND_corpus.py:179-213', 'exec')
    cases, H, C = graph_cases()
    for cats in cases:
        g_ref, m_ref, i_ref = run_reference_graph(code, cats, H, C, flags)
        g, m, i = G.build_history_graph(cats, H, C, **flags)
        assert g.dtype == g_ref.dtype == np.float32
        assert np.array_equal(g, g_ref), (flags, cats)
        assert np.array_equal(m, m_ref) and np.array_equal(i, i_ref)
    # MIND-shaped size as well
    rng = np.random.default_rng(5)
    for _ in range(6):
        cats = list(rng.integers(0, 18, size=int(rng.integers(1, 51))))
        g_ref, m_ref, i_ref = run_reference_graph(code, cats, 50, 18, flags)
        g, m, i = G.build_history_graph(cats, 50, 18, **flags)
        assert np.array_equal(g, g_ref) and np.array_equal(m, m_ref) and np.array_equal(i, i_ref)


def test_graph_restatement_matches_committed_reference_vectors():
    """tests/golden/graph_flags.npz = outputs of the executed reference source (make_golden.py graph_flags)"""
    z = np.load(os.path.join(GOLDEN_DIR, 'graph_flags.npz'))
    cases, H, C = graph_cases()
    for fi, flags in enumerate(FLAG_SETS):
        for ci, cats in enumerate(cases):
            g, m, i = G.build_history_graph(cats, H, C, **flags)
            assert np.array_equal(g, z['graph_%d' % fi][ci]), (flags, cats)
            assert np.array_equal(m, z['mask_%d' % fi][ci]) and np.array_equal(i, z['idx_%d' % fi][ci])


def metric_cases(seed=7, n=25):
    rng = np.random.default_rng(seed)
    labels, scores = [], []
    for k in range(n):
        c = int(rng.integers(2, 40))
        s = rng.normal(size=c).astype(np.float32)
        if k % 3 == 0:
            s = np.round(s * 2) / 2                       # ties: the stable sort of util.py:57 decides
        lab = np.zeros(c, dtype=np.int64)
        lab[rng.choice(c, size=int(rng.integers(1, max(2, c // 3))), replace=False)] = 1
        if lab.sum() == c:
            lab[0] = 0
        labels.append(lab.tolist())
        scores.append([float(x) for x in s])
    return labels, scores


def reference_rank_lines():
    """util.py:58-61: the per-impression ranking (sort by score, descending, Python's stable sort)"""
    with open(os.path.join(R.REFERENCE_ROOT, 'util.py')) as f:
        lines = f.readlines()
    body = ''.join(lines[57:61])
    assert 'sub_score.sort(key=lambda x: x[0], reverse=True)' in body
    return textwrap.dedent(body)


def reference_metrics(labels, scores):
    spec = importlib.util.spec_from_file_location('_ref_evaluate', os.path.join(R.REFERENCE_ROOT, 'evaluate.py'))
    ev = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ev)
    code = compile(reference_rank_lines(), 'util.py:58-61', 'exec')
    truth, sub, all_ranks = io.StringIO(), io.StringIO(), []
    for k, (lab, sc) in enumerate(zip(labels, scores)):
        env = dict(sub_score=[[s, j] for j, s in enumerate(sc)])                 # util.py:53-54 builds [score, index] pairs
        exec(code, env)                                                          # util.py:58-61: sub_score -> result
        all_ranks.append(list(env['result']))
        truth.write('%d %s\n' % (k + 1, json.dumps(lab).replace(' ', '')))
        sub.write('%d %s\n' % (k + 1, str(env['result']).replace(' ', '')))     # util.py:61
    truth.seek(0)
    sub.seek(0)
    return ev.scoring(truth, sub), all_ranks


@needs_reference
def test_metrics_restatement_equals_live_evaluate_py():
    labels, scores = metric_cases()
    ref, ref_ranks = reference_metrics(labels, scores)
    for k, sc in enumerate(scores):
        assert OM.ranks_from_scores(sc) == ref_ranks[k]
    mine = OM.scoring(labels, scores)
    for a, b in zip(ref, mine):
        assert abs(float(a) - float(b)) < 1e-12


def test_metrics_restatement_matches_committed_reference_vectors():
    z = np.load(os.path.join(GOLDEN_DIR, 'metrics.npz'))
    labels, scores = metric_cases()
    mine = OM.scoring(labels, scores)
    assert np.allclose(np.array(mine, dtype=np.float64), z['metrics'], rtol=0, atol=1e-12)
    flat = np.concatenate([np.array(OM.ranks_from_scores(sc)) for sc in scores])
    assert np.array_equal(flat, z['ranks'])


@needs_reference
@pytest.mark.parametrize('over', [dict(gcn_layer_norm=True), dict(no_gcn_residual=True), dict(gcn_layer_norm=True, no_gcn_residual=True)],
                         ids=['layer_norm', 'no_residual', 'layer_norm+no_residual'])
def test_oracle_gcn_flags_match_live_reference(over):
    cfg = O.make_config(vocabulary_size=300, max_history_num=6, max_title_length=8, max_abstract_length=12, subCategory_num=20,
                        gcn_layer_num=3, dropout_rate=0.0, **over)
    from nnr_b200.synthetic import SyntheticMIND
    syn = SyntheticMIND(news_num=100, vocabulary_size=300, subCategory_num=20, max_title_length=8, max_abstract_length=12,
                        max_history_num=6, lengths='uniform', seed=2)
    batch = syn.batch(3, seed=4)
    p = O.formula_params(cfg, salt=1)
    m = R.build_reference_model(cfg, p)
    m.train()
    ref = R.run_reference(m, batch, sort_fn=O.stable_sort)
    O.loss_fn(ref).backward()
    logits, loss, grads = O.forward_backward(p, cfg, batch, sort_fn=O.stable_sort)
    assert (ref.detach() - logits).abs().max().item() < 5e-6
    named = dict(m.named_parameters())
    gmax = max(float(named[k].grad.abs().max()) for k in grads if named[k].grad is not None)
    for k, g in grads.items():
        rg = named[k].grad
        rg = torch.zeros_like(g) if rg is None else rg
        # two fp32 implementations (the reference's packed ATen LSTM vs the oracle's explicit loop): rounding-level agreement,
        # measured against the tensor's own scale or 1 % of the largest gradient entry of the model, whichever is larger
        assert (rg - g).abs().max().item() <= 2e-5 * max(rg.abs().max().item(), 1e-2 * gmax), k
