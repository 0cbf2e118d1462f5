"""Cost of the hidden size: for each hidden_dim, one JSON line with
  - the bidirectional LSTM forward and BPTT alone at the BASELINE config-2 history shape (N = 3520 rows, L = 128, MIND-like
    lengths), CUDA events over warmed-up repeats;
  - the captured TrainStep at BASELINE config 2 (bench.py defaults) with that hidden_dim: ms/step and impressions/s;
  - the GPU name and power limit, read in the same run.

usage: python scripts/hidden_dim_sweep.py [--hidden 64 100 128 160 200] [--steps 20] [--warmup 5]"""
import argparse, json, math, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
import nnr_b200
from nnr_b200 import ops
from nnr_b200.synthetic import SyntheticMIND, batch_args
from nnr_b200.trainer import TrainStep


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'], capture_output=True,
                           text=True, timeout=30)
        power = q.stdout.strip() or None
    except Exception:
        power = None
    return name, power


def time_ms(fn, reps):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def lstm_ms(Hd, dev, N=3520, L=128, reps=10):
    g = torch.Generator().manual_seed(0)
    lens = torch.exp(torch.randn(N, generator=g) * 0.8 + math.log(40.0) - 0.32).round().clamp_(1, L).long()
    lens[: N // 50] = L
    ntok = int(lens.sum())
    len_ = lens.to(torch.int32).to(dev)
    off = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(torch.int32).to(dev)
    order = torch.sort(lens, descending=True, stable=True)[1].to(torch.int32).to(dev)
    gx0 = torch.randn(ntok, 8 * Hd, generator=g).to(dev) * 0.5
    gx = gx0.clone()
    w_hh = (torch.randn(2, 4 * Hd, Hd, generator=g) / math.sqrt(Hd)).to(dev)
    h, cst = torch.empty(ntok, 2 * Hd, device=dev), torch.empty(ntok, 2 * Hd, device=dev)
    cn = torch.empty(N, 2 * Hd, device=dev)
    dh, dcn = torch.randn(ntok, 2 * Hd, device=dev) * 0.1, torch.randn(N, 2 * Hd, device=dev) * 0.1
    fwd = time_ms(lambda: ops.lstm_fwd(gx, w_hh, len_, off, order, N, L, Hd, h, cst, cn), reps)
    gx.copy_(gx0)
    ops.lstm_fwd(gx, w_hh, len_, off, order, N, L, Hd, h, cst, cn)
    stash = gx.clone()

    def bwd():
        gx.copy_(stash)                       # BPTT overwrites the stash with dL/dgx
        ops.lstm_bwd(gx, cst, w_hh, len_, off, order, N, L, Hd, dh, dcn)
    copy = time_ms(lambda: gx.copy_(stash), reps)
    return fwd, time_ms(bwd, reps) - copy, ntok


def step_ms(Hd, dev, steps, warmup):
    sys.argv = [sys.argv[0]]
    a = bench.parse()
    cfg = bench.make_config(a)
    cfg.hidden_dim = Hd
    syn = SyntheticMIND(news_num=20000, vocabulary_size=a.vocab, lengths=a.lengths, seed=0)
    cfg.pretrained_word_embedding = syn.word_table()
    model = nnr_b200.Model(cfg); model.initialize(); model.to(dev)
    ts = TrainStep(model, lr=1e-4, gradient_clip_norm=4.0, cuda_graph=True)
    devb = [batch_args(syn.batch(a.batch, seed=i), dev) for i in range(4)]
    for i in range(warmup):
        ts.step(*devb[i % 4])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        ts.step(*devb[i % 4])
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return ms, a.batch * 1e3 / ms, a.batch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--hidden', type=int, nargs='+', default=[64, 100, 128, 160, 200])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    args = ap.parse_args()
    dev = torch.device('cuda:0')
    name, power = gpu_info()
    for Hd in args.hidden:
        f, b, ntok = lstm_ms(Hd, dev)
        ms, ips, batch = step_ms(Hd, dev, args.steps, args.warmup)
        print(json.dumps({'hidden_dim': Hd, 'cluster_ctas': max(2, (Hd + 39) // 40),
                          'lstm_shape': {'N': 3520, 'L': 128, 'tokens': ntok, 'lengths': 'mind'},
                          'lstm_fwd_ms': round(f, 4), 'lstm_bptt_ms': round(b, 4),
                          'train_step': {'config': 'BASELINE config 2', 'impressions_per_step': batch, 'cuda_graph': True,
                                         'steps': args.steps, 'warmup': args.warmup},
                          'ms_per_step': round(ms, 3), 'impressions_per_s': round(ips, 1),
                          'gpu': name, 'power_limit': power}), flush=True)
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
