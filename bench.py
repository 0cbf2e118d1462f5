"""bench.py -- CNE+SUE training-step throughput on B200 (BASELINE.json metric: train impressions/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference ...                      # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's results as .npy

One "step" = the hot path of reference trainer.py:105-120 over one batch of 64 synthetic
MIND-shaped impressions per GPU (title <= 32, abstract <= 128, history 50, K = 4, 300-d words,
gcn_layer_num 4, dropout 0.2, V = 40 000): forward, loss, backward, clip_grad_norm_(4), Adam.
N > 1: one process per GPU (torchrun), every rank its own batches (weak scaling), one NCCL
all-reduce of the flat gradient buffer per step.  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = 'cne_sue_train_impressions_per_sec'
UNIT = 'impressions/s'


def load_synthetic():
    """nnr_b200/synthetic.py (numpy / torch-CPU only) loaded by path: importing it as ``nnr_b200.synthetic`` would run
    the package __init__ and dlopen libnnr_b200.so, which the CPU reference arm must not touch"""
    import importlib.util
    spec = importlib.util.spec_from_file_location('_nnr_synthetic_standalone', os.path.join(ROOT, 'nnr_b200', 'synthetic.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='nnr_b200', choices=['nnr_b200', 'reference'])
    ap.add_argument('--batch', type=int, default=64, help='impressions per GPU per step')
    ap.add_argument('--vocab', type=int, default=40000)
    ap.add_argument('--lengths', default='mind', choices=['mind', 'full', 'uniform'])
    ap.add_argument('--dropout', type=float, default=0.2)
    ap.add_argument('--cpu-sample', type=int, default=16, help='impressions per step of the bounded CPU-baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-profile', action='store_true', help='skip the per-op CUDA-event breakdown')
    ap.add_argument('--gemm-detail', action='store_true', help='print the per-shape GEMM table to stderr')
    ap.add_argument('--dtype', default='f32', choices=['f32', 'bf16'],
                    help='f32: fp32-grade arithmetic (split-operand tensor-core products); bf16: the reduced-precision variant of '
                         'BASELINE config 4 (one 16-bit product per GEMM and per recurrent step, fp32 accumulation)')
    ap.add_argument('--sharding', default='balanced', choices=['balanced', 'random'],
                    help='N > 1: how the global batch is cut into per-rank shards (balanced = equal token counts per rank and step)')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel of a step from the host instead of replaying a CUDA graph')
    ap.add_argument('--no-extras', action='store_true', help='skip the extra measurements (scoring, full-length regime)')
    ap.add_argument('--scoring-news', type=int, default=100000, help='news in the synthetic corpus of the scoring extra')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (loss, gradient norm before clipping, every '
                         'parameter after the update and its gradient before clipping) to DIR/<name>.npy, to compare two builds '
                         'output for output')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs writes the results of the CUDA path; --impl reference has none')
    return a


def workload_name(a):
    return 'cne_sue_train_step_b%d_k4_h50_t32_a128_e300_v%d_gcn4_%s_lengths' % (a.batch, a.vocab, a.lengths)


def make_config(a):
    from types import SimpleNamespace
    return SimpleNamespace(word_embedding_dim=300, vocabulary_size=a.vocab, word_threshold=3, tokenizer='MIND',
                           max_title_length=32, max_abstract_length=128, dataset='synthetic', category_num=18,
                           subCategory_num=285, category_embedding_dim=50, subCategory_embedding_dim=50,
                           dropout_rate=a.dropout, hidden_dim=200, attention_dim=200, gcn_layer_num=4,
                           no_gcn_residual=False, gcn_layer_norm=False, max_history_num=50, news_encoder='CNE',
                           user_encoder='SUE', click_predictor='dot_product', negative_sample_num=4)


# -------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks line"), NVML in a thread
# -------------------------------------------------------------------------------------------------
class Clocks:
    def __init__(self, index):
        self.samples, self.reasons, self.stop = [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        nv = self.nv
        names = {'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40,
                 'hw_power_brake': 0x80}
        while not self.stop:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.nv:
            self.t.join(timeout=1)

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


# -------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference, bounded sample, all host threads
# -------------------------------------------------------------------------------------------------
def cpu_dropout_masks(cfg, batch, p, gen):
    """keep-masks (0 or 1/(1-p)) for the seven dropout sites of the reference CNE+SUE (newsEncoders.py:53,117-118,
    userEncoders.py:80,91, layers.py:320-322; GCN inter-layer rate = p/2), drawn on the CPU like nn.Dropout does"""
    def keep(shape, rate):
        return torch.bernoulli(torch.full(shape, 1.0 - rate), generator=gen) / (1.0 - rate)
    B, n = batch['news_title_text'].shape[:2]
    H = batch['user_title_text'].shape[1]
    E, T, A = cfg.word_embedding_dim, cfg.max_title_length, cfg.max_abstract_length
    D = 4 * cfg.hidden_dim + cfg.category_embedding_dim + cfg.subCategory_embedding_dim
    C = cfg.category_num

    def cne(N, Bn, nn_):
        return {'title': keep((N, T, E), p), 'content': keep((N, A, E), p),
                'category': keep((Bn, nn_, cfg.category_embedding_dim), p), 'subCategory': keep((Bn, nn_, cfg.subCategory_embedding_dim), p)}
    sue = {'proxy': keep((B, C, D), p), 'cluster': keep((B, n, C + 1, D), p)}
    for l in range(cfg.gcn_layer_num - 1):
        sue['gcn%d' % l] = keep((B, H + C, D), p / 2.0)
    return {'news': cne(B * n, B, n), 'history': cne(B * H, B, H), 'sue': sue}


def cpu_train_step_rate(a, sample, steps, warmup):
    """`warmup` untimed + EXACTLY `steps` timed training steps (forward, loss, backward, clip_grad_norm_(4), Adam) of the
    oracle port on `sample` impressions per step, same shapes / vocabulary / length regime / dropout as the GPU arm,
    all host threads.  Returns (impressions/s, cores, seconds per step)."""
    from oracle import nnr_oracle as O
    syn_mod = load_synthetic()
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    cfg = O.make_config(vocabulary_size=a.vocab, dropout_rate=a.dropout)
    syn = syn_mod.SyntheticMIND(news_num=20000, vocabulary_size=a.vocab, lengths=a.lengths, seed=0)
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(1)
    p = {k: (torch.randn(s) * 0.05) for k, s in O.param_shapes(cfg).items()}
    p['news_encoder.word_embedding.weight'] = syn.word_table()
    state = {}
    times = []
    for i in range(warmup + steps):
        batch = syn.batch(sample, seed=100 + i)
        t0 = time.perf_counter()
        masks = cpu_dropout_masks(cfg, batch, a.dropout, gen) if a.dropout > 0 else None
        _, loss, grads = O.forward_backward(p, cfg, batch, lstm_impl='aten', dropout_masks=masks)   # ATen packed LSTM = reference path
        O.clip_and_adam(p, grads, state, i + 1)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    return sample / t, cores, t


def cpu_sample_note(a, sample, steps, warmup, t):
    return ('%d impressions per step (a bounded sample of the %d-impression batch; same shapes, vocabulary, length regime and '
            'dropout %.2f), %d warm-up + %d timed train steps (fwd+bwd+clip+Adam) of the oracle port with the packed ATen LSTM, '
            '%.2f s per step' % (sample, a.batch, a.dropout, warmup, steps, t))


def run_reference(a):
    """--impl reference: the reference's CPU path (oracle port; the reference is Python and cannot travel to the GPU box),
    EXACTLY --steps timed and --warmup untimed steps, each on --cpu-sample impressions.  Imports neither the nnr_b200
    package nor its shared library."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    sample = a.cpu_sample
    rate, cores, t = cpu_train_step_rate(a, sample, steps=a.steps, warmup=a.warmup)
    line = {'metric': METRIC, 'value': rate, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': t * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'impl': 'reference',
            'config': {'workload': workload_name(a), 'impressions_per_step': sample, 'dropout': a.dropout,
                       'note': 'CPU only: oracle port of the reference PyTorch path; each step is a bounded %d-impression '
                               'sample of the workload (value is impressions/s, i.e. batch-normalised)' % sample},
            'cpu_baseline': {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                             'sample': cpu_sample_note(a, sample, a.steps, a.warmup, t)},
            'e2e': {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------
# extra measurements printed on the same JSON line (N = 1 only)
# -------------------------------------------------------------------------------------------------
CNE_FWD_FLOP_PER_TOKEN = 960000 + 640000 + 320000 + 160000 + 800      # SURVEY 8d: W_ih, recurrent, gate, self-attn affine, folded cross scores


def extra_scoring(a, cfg, model, dev, peaks):
    """BASELINE config 3 / metric "scoring news-enc/sec" (reference path util.py:10-68): encode a synthetic corpus once
    with the CNE kernels (eval), then SUE + click scores of impressions against the cached corpus."""
    from nnr_b200.scoring import CorpusScorer
    from nnr_b200.synthetic import SyntheticMIND
    news, impressions, cands, chunk, batch = a.scoring_news, 4096, 37, 4096, 256
    syn = SyntheticMIND(news_num=news, vocabulary_size=a.vocab, lengths=a.lengths, seed=5)
    was_training = model.training
    sc = CorpusScorer(model, syn.news_title_text, syn.news_title_mask, syn.news_abstract_text, syn.news_abstract_mask,
                      syn.news_category, syn.news_subCategory, chunk=chunk)
    sc.encode_corpus()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        sc.encode_corpus()
    e1.record()
    torch.cuda.synchronize()
    enc_ms = e0.elapsed_time(e1) / reps
    hist, hl, cand = syn.sample_behaviors(impressions, news_num=cands, seed=1)
    hist, hl, cand = torch.from_numpy(hist).to(dev), torch.from_numpy(hl).to(dev), torch.from_numpy(cand).to(dev)

    def run():
        out = None
        for i in range(0, impressions, batch):
            out = sc.score(hist[i:i + batch], hl[i:i + batch], cand[i:i + batch])
        return out
    run()
    torch.cuda.synchronize()
    e0.record()
    out = run()
    e1.record()
    torch.cuda.synchronize()
    sc_ms = e0.elapsed_time(e1)
    tokens = int(syn.title_len.sum() + syn.abstract_len.sum())
    tflops = tokens * CNE_FWD_FLOP_PER_TOKEN / (enc_ms * 1e-3) / 1e12
    if was_training:
        model.train()
    return {'metric': 'cne_scoring_news_enc_per_sec', 'value': news / (enc_ms * 1e-3), 'unit': 'news/s', 'encode_ms': enc_ms,
            'corpus_news': news, 'corpus_tokens': tokens, 'tokens_per_sec': tokens / (enc_ms * 1e-3), 'chunk': chunk,
            'scored_impressions_per_sec': impressions / (sc_ms * 1e-3), 'candidates_per_impression': cands, 'history': 50,
            'score_ms': sc_ms, 'finite': bool(torch.isfinite(out).all()),
            'roofline': {'bound': 'tensor', 'achieved': tflops, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': tflops / peaks['bf16_tflops'],
                         'mma_per_algorithmic_flop': 3, 'frac_of_peak_in_issued_mma': 3 * tflops / peaks['bf16_tflops'], 'traffic': None,
                         'note': 'whole CNE forward (all kernels of encode_corpus): %d algorithmic flop per valid token (SURVEY 8d) / wall time'
                                 % CNE_FWD_FLOP_PER_TOKEN}}


def extra_full_lengths(a, ts, dev, peaks):
    """the roofline worst case of SURVEY 8d: every title has 32 and every abstract 128 valid tokens (563 200 tokens per step)"""
    from nnr_b200 import profiler
    from nnr_b200.synthetic import SyntheticMIND, batch_args
    syn = SyntheticMIND(news_num=20000, vocabulary_size=a.vocab, lengths='full', seed=0)
    devb = [batch_args(syn.batch(a.batch, seed=50 + i), dev) for i in range(2)]
    for i in range(3):
        ts.step(*devb[i % 2])
    torch.cuda.synchronize()
    steps = 5
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        ts.step(*devb[i % 2])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    ts._eager_step(*devb[1])
    torch.cuda.synchronize()
    with profiler.capture() as prof:
        ts._eager_step(*devb[0])
        torch.cuda.synchronize()
    bd = prof.summary(steps=1)
    out = {'workload': workload_name(a).replace('%s_lengths' % a.lengths, 'full_lengths'), 'value': a.batch / (ms * 1e-3), 'unit': UNIT,
           'ms_per_step': ms, 'steps': steps, 'warmup': 3, 'tokens_per_step': a.batch * 55 * 160}
    rows = {r['kernel']: r for r in profiler.roofline_table(bd, ROOT)}
    for k in ('gemm_tc_kernel', 'lstm_fwd', 'lstm_bwd', 'embed_gather_fwd', 'embed_gather_bwd', 'attn_pool_fwd', 'attn_pool_bwd'):
        if k in rows:
            out[k] = {kk: rows[k][kk] for kk in ('ms', 'achieved', 'unit', 'frac') if kk in rows[k]}
            if 'frac_of_peak_in_issued_mma' in rows[k]:
                out[k]['frac_of_peak_in_issued_mma'] = rows[k]['frac_of_peak_in_issued_mma']
    return out


# -------------------------------------------------------------------------------------------------
# --dump-outputs: the results of the last timed step, for comparing two builds output for output
# -------------------------------------------------------------------------------------------------
DUMP_MAX_ELEMENTS = 1 << 18      # per tensor; keeps the directory under 40 MB (the word table is the only tensor --vocab resizes)


def dump_outputs(directory, ts, loss):
    """What a caller of TrainStep.step has after the last timed step: the returned loss, the total gradient norm before
    clipping (ts.grad_norm, what clip_grad_norm_ returns) and, for every trainable parameter, its value after the Adam update
    (param.<name>) and its gradient before clipping (grad.<name>; with N > 1 the sum over ranks, which the optimizer kernel
    scales by 1/N), flattened, float32.  A tensor of more than DUMP_MAX_ELEMENTS elements is written as its
    elements at DUMP_MAX_ELEMENTS sorted flat positions drawn by a generator seeded with 0: the same positions on every run
    and every build."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    torch.cuda.synchronize()
    out = {'loss': loss.detach(), 'grad_norm': ts.grad_norm}
    for name, p in ts.model.named_parameters():
        if p.requires_grad:
            out['param.' + name] = p.detach()
            out['grad.' + name] = p.grad
    for name, t in out.items():
        a = t.float().reshape(-1).cpu().numpy()
        if a.size > DUMP_MAX_ELEMENTS:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))]
        np.save(os.path.join(directory, name + '.npy'), a)


def main():
    a = parse()
    if a.impl == 'reference':
        return run_reference(a)
    if a.dtype == 'bf16':
        os.environ['NNR_GEMM_ALGO'] = 'bf16'                  # read once by libnnr_b200.so: GEMMs and the LSTM recurrence
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    import nnr_b200
    from nnr_b200 import ops
    from nnr_b200.synthetic import SyntheticMIND, batch_args, FIELDS
    from nnr_b200.trainer import PackedBatch, TrainStep

    cfg = make_config(a)
    syn = SyntheticMIND(news_num=20000, vocabulary_size=a.vocab, lengths=a.lengths, seed=0)
    cfg.pretrained_word_embedding = syn.word_table()
    torch.manual_seed(1234)                                   # same init on every rank (main.py:14-15,24)
    model = nnr_b200.Model(cfg)
    model.initialize()
    model.to(dev)
    ts = TrainStep(model, lr=1e-4, gradient_clip_norm=4.0, world_size=world, cuda_graph=not a.no_graph)
    torch.manual_seed(1000 + rank)                            # dropout streams differ per rank

    nb = 4                                                    # distinct batches per rank, rotated
    if world == 1 or a.sharding == 'random':
        host = [syn.batch(a.batch, seed=7 * rank + i) for i in range(nb)]
    else:
        # token-balanced sharding (trainer.balanced_shards): every rank draws the same global batch of world x batch
        # impressions (like the reference, where every rank runs the same sampling with the same seed, trainer.py:255-258) and
        # takes the shard a greedy longest-first assignment gives it, so that all ranks have the same number of tokens per step
        from nnr_b200.trainer import balanced_shards
        import numpy as np
        host = []
        for i in range(nb):
            # the global batch = exactly the impressions the ranks would draw on their own (--sharding random), re-dealt
            parts = [syn.sample_behaviors(a.batch, seed=7 * r + i) for r in range(world)]
            hist, hl, cand = (np.concatenate([p[j] for p in parts]) for j in range(3))
            per_news = (syn.title_len + syn.abstract_len)
            cost = per_news[hist].sum(1) + per_news[cand].sum(1)
            idx = np.asarray(balanced_shards(cost, world)[rank])
            host.append(syn.materialize(hist[idx], hl[idx], cand[idx]))
    for b in host:
        for k in FIELDS:
            if torch.is_tensor(b[k]):
                b[k] = b[k].contiguous().pin_memory()
    devb = [batch_args(b, dev) for b in host]
    # one contiguous buffer per batch: device-resident for `value`, pinned host memory for `e2e` (what a collate_fn +
    # pin_memory worker hands over); a step is then ONE copy into the captured graph's input buffer + one graph launch
    devp = [PackedBatch.pack(b, device=dev) for b in devb]
    hostp = [PackedBatch.pack(batch_args(b), pin=True) for b in host]
    tok = sum(int(b['user_title_mask'].sum() + b['user_content_mask'].sum() + b['news_title_mask'].sum()
                  + b['news_content_mask'].sum()) for b in host) / nb
    slots = a.batch * 55 * 160
    h2d = hostp[0].flat.numel()

    def fresh(args):   # masks are mutated in place by the model (like the reference): idempotent, reuse is safe
        return args

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing -------------------------------------------------------------
    for i in range(a.warmup):
        ts.step(devp[i % nb])
    barrier()
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with Clocks(local_rank) as clk:
        e0.record()
        for i in range(a.steps):
            loss = ts.step(devp[i % nb])
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.launch_count() - launches0
    if ts.cuda_graph:            # kernels of this library inside one replayed graph (counted while it was captured) x replays
        launches = a.steps * max(ts.launches_per_graph.values())
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    value = a.batch * world * a.steps / (ms / 1e3)
    if a.dump_outputs and rank == 0:                          # before the passes below move the parameters on
        dump_outputs(a.dump_outputs, ts, loss)

    # ---- end to end: pinned host batch -> device every step, loss read back every step ----------
    for i in range(2):                                        # untimed warm-up of this path (allocator, copy engine)
        ts.step(ts.prefetch(hostp[i % nb])).item()
    barrier()
    from nnr_b200.trainer import LossLog

    def run_e2e(blocking):
        """K steps from pinned host batches; every step's inputs cross PCIe inside the timed region and every step's loss is
        read back to the host: blocking = float(loss) before the next step is enqueued (reference trainer.py:115);
        otherwise through trainer.LossLog (pinned slot + event, consumed while the next step runs; all K values read
        before the end).  The next batch's host-to-device copy is enqueued on a copy stream before the host waits for
        anything (what a pinned-memory DataLoader gives the reference)."""
        log = LossLog()
        vals = []
        e0.record()
        nxt = ts.prefetch(hostp[0])                           # inside the timed region: every step's batch is copied H2D
        for i in range(a.steps):
            cur = nxt
            loss = ts.step(cur)
            if not blocking:
                vals += log.push(loss, weight=a.batch)
            if i + 1 < a.steps:
                nxt = ts.prefetch(hostp[(i + 1) % nb])
            if blocking:
                vals.append(loss.item())
        vals += log.drain()
        e1.record()
        barrier()
        assert len(vals) == a.steps
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return a.batch * world * a.steps / (t.item() / 1e3), vals[-1]

    e2e_blocking, _ = run_e2e(True)
    e2e, loss_host = run_e2e(False)

    # ---- end to end, index-only batches (SURVEY 8f-1): the tokenised corpus lives in HBM; per step only the
    # history / candidate ids cross PCIe, the 21 model inputs are gathered and the graph is built on the device ------
    from nnr_b200.corpus import DeviceCorpus
    corpus = DeviceCorpus.from_synthetic(syn, dev)
    ids_host = [tuple(h[k].contiguous().pin_memory() for k in ('history_ids', 'history_len', 'candidate_ids')) for h in host]
    ids_bytes = sum(v.numel() * v.element_size() for v in ids_host[0])
    for i in range(2):
        ts.step_ids(corpus, *ids_host[i % nb])
    barrier()
    e0.record()
    log = LossLog()
    n_read = 0
    for i in range(a.steps):
        loss = ts.step_ids(corpus, *ids_host[i % nb])
        n_read += len(log.push(loss, weight=a.batch))
    n_read += len(log.drain())
    assert n_read == a.steps
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ids = a.batch * world * a.steps / (t.item() / 1e3)

    # ---- N > 1: what the scaling loss is made of: the collective alone, and the spread of the ranks' compute time ----------
    scaling_detail = None
    if world > 1:
        barrier()
        reps = 5
        e0.record()
        for _ in range(reps):
            dist.all_reduce(ts.gflat, op=dist.ReduceOp.SUM)
        e1.record()
        barrier()
        coll_all = e0.elapsed_time(e1) / reps
        a_t, b_t = ts.stage_bounds['table']
        e0.record()
        for _ in range(reps):
            dist.all_reduce(ts.gflat[a_t:b_t], op=dist.ReduceOp.SUM)
        e1.record()
        barrier()
        coll_table = e0.elapsed_time(e1) / reps
        ts.world_size = 1                                     # compute only: no collective, host-launched, per rank
        for i in range(2):
            ts._eager_step(*fresh(devb[i % nb]))
        torch.cuda.synchronize()
        e0.record()
        for i in range(a.steps):
            ts._eager_step(*fresh(devb[i % nb]))
        e1.record()
        torch.cuda.synchronize()
        ts.world_size = world
        mine = torch.tensor([e0.elapsed_time(e1) / a.steps], device=dev)
        allms = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allms, mine)
        allms = [float(x.item()) for x in allms]
        # every rank changed its replica independently: restore identical parameters before anything else uses them
        dist.broadcast(ts.flat, 0)
        dist.broadcast(ts.exp_avg, 0)
        dist.broadcast(ts.exp_avg_sq, 0)
        ts._refresh_weight_planes()
        scaling_detail = {'allreduce_whole_flat_buffer_ms': coll_all, 'allreduce_table_slice_ms': coll_table,
                          'flat_buffer_bytes': ts.gflat.numel() * 4, 'table_slice_bytes': (b_t - a_t) * 4,
                          'compute_only_ms_per_rank': allms, 'rank_skew_ms': max(allms) - sum(allms) / len(allms),
                          'note': 'the collective alone (back to back after a barrier; the table slice is the part the step cannot '
                                  'overlap), and each rank\'s host-launched step without any collective: a step of the job takes '
                                  'max over ranks + the exposed part of the collective'}

    # ---- per-op breakdown with CUDA events (dominant kernel -> roofline) ---------------------------
    roofline = None
    roofline_table = None
    breakdown = None
    if not a.no_profile:
        # every rank runs the two extra steps (they contain the gradient all-reduce); only rank 0 records events
        from nnr_b200 import profiler
        for i in range(2):                                    # host-launched warm-up (fills the eager allocator pool)
            ts._eager_step(*fresh(devb[i % nb]))
        torch.cuda.synchronize()
        if rank == 0:
            with profiler.capture() as prof:              # per-op events need host launches: the same step, not replayed
                for i in range(2):
                    ts._eager_step(*fresh(devb[i % nb]))
                torch.cuda.synchronize()
            breakdown = prof.summary(steps=2)
            if a.gemm_detail:
                for k, v in prof.detail.items():
                    print('%-44s %8.3f ms  %4.1f calls  %7.1f TFLOP/s' % (k, v['ms'], v['calls'], v['tflops']), file=sys.stderr)
            roofline = profiler.roofline(breakdown, tokens_per_step=tok, batch=a.batch, root=ROOT)
            roofline_table = profiler.roofline_table(breakdown, ROOT)
        else:
            for i in range(2):
                ts._eager_step(*fresh(devb[i % nb]))
            torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if rank != 0:
        return finish(ts, world)

    cpu = None
    if not a.no_cpu_baseline and world == 1:
        rate, cores, tcpu = cpu_train_step_rate(a, a.cpu_sample, steps=3, warmup=1)
        cpu = {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': cpu_sample_note(a, a.cpu_sample, 3, 1, tcpu)}
    extra = {}
    if world == 1 and not a.no_extras:
        from nnr_b200 import profiler as _prof
        peaks = _prof.measured_peaks(ROOT)
        extra['full_lengths'] = extra_full_lengths(a, ts, dev, peaks)
        extra['scoring'] = extra_scoring(a, cfg, model, dev, peaks)
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': ms / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': a.dtype, 'data': 'synthetic',
            'config': {'workload': workload_name(a), 'global_batch': a.batch * world, 'parallelism': 'dp%d' % world,
                       'sharding': ('n/a (one rank)' if world == 1 else
                                    'token-balanced: every rank draws the same global batch and takes the shard of a greedy longest-first '
                                    'assignment over the impressions\' token counts (nnr_b200.trainer.balanced_shards)'
                                    if a.sharding == 'balanced' else 'random shards (independent batches per rank)'),
                       'valid_token_fraction': tok / slots, 'tokens_per_step_per_gpu': tok,
                       'l2_policy': 'per-step working set (activations+stashes, GBs) >> 126 MB L2; %d rotating batches' % nb,
                       'launch': 'cuda graph replay (one launch per step)' if ts.cuda_graph else 'host launches',
                       'arithmetic': ('bf16 variant: one 16-bit product per GEMM / recurrent step, fp32 accumulation, fp32 activations; '
                                      'logits within 2e-2, gradients within 5e-2 of the fp64 reference per tensor (tests/test_model_gpu.py)')
                       if a.dtype == 'bf16' else 'fp32-grade: split 16-bit operands, 3 tensor-core products per flop',
                       'loss': loss_host},
            'clocks': clk.summary(),
            'e2e': {'value': e2e, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                    'loss_read': 'every step, pinned non-blocking D2H + event (trainer.LossLog), consumed while the next step '
                                 'runs; all K losses are on the host before the timed region ends',
                    'value_blocking_loss_read': e2e_blocking},
            'e2e_index_only': {'value': e2e_ids, 'unit': UNIT, 'h2d_bytes_per_step': ids_bytes, 'd2h_bytes_per_step': 4,
                               'corpus_bytes_resident': corpus.nbytes(),
                               'note': 'nnr_b200.corpus.DeviceCorpus + TrainStep.step_ids: ids in, batch gathered and graph built on the device'},
            'gpu_launches': int(launches), 'scaling_detail': scaling_detail,
            'roofline': roofline, 'roofline_by_kernel': roofline_table, 'cpu_baseline': cpu, 'extra': extra,
            'breakdown_ms_per_step': breakdown}
    print(json.dumps(line))
    finish(ts, world)


def finish(ts, world):
    """N > 1: leave without tearing the NCCL communicator down -- destroying a process group whose collectives were captured
    in CUDA graphs waits for minutes (measured: the first 2-GPU run of this round printed its line and then sat in
    destroy_process_group until the driver's limit); the graphs are released first and every rank exits after a last barrier"""
    if world <= 1:
        return
    ts._graphs.clear()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
