"""Micro-benchmark of the persistent LSTM kernels: time per tile-step from uniform-length batches.

usage: python scripts/lstm_bench.py [--hidden 200 128 ...]   (hidden sizes to time, default 200)"""
import argparse, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from nnr_b200 import ops

ap = argparse.ArgumentParser()
ap.add_argument('--hidden', type=int, nargs='+', default=[200], help='hidden sizes (hidden_dim) to time')
args = ap.parse_args()
dev = torch.device('cuda:0')
for Hd in args.hidden:
    if len(args.hidden) > 1:
        print('hidden_dim %d' % Hd, flush=True)
    for (N, L) in [(32, 64), (1024, 64), (2048, 64), (4096, 32), (3520, 128)]:
        lens = torch.full((N,), L, dtype=torch.int32, device=dev)
        off = (torch.arange(N + 1, device=dev) * L).to(torch.int32)
        order = torch.arange(N, dtype=torch.int32, device=dev)
        gx = torch.randn(N * L, 8 * Hd, device=dev) * 0.1
        w_hh = torch.randn(2, 4 * Hd, Hd, device=dev) * 0.05
        h = torch.empty(N * L, 2 * Hd, device=dev)
        cst = torch.empty(N * L, 2 * Hd, device=dev)
        cn = torch.empty(N, 2 * Hd, device=dev)
        dh = torch.randn(N * L, 2 * Hd, device=dev) * 0.1
        dcn = torch.randn(N, 2 * Hd, device=dev) * 0.1
        for name, fn in (('fwd', lambda: ops.lstm_fwd(gx, w_hh, lens, off, order, N, L, Hd, h, cst, cn)),
                         ('bwd', lambda: ops.lstm_bwd(gx, cst, w_hh, lens, off, order, N, L, Hd, dh, dcn))):
            fn(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); fn(); e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 2
            tiles = (N + 31) // 32 * 2
            waves = max(1.0, tiles / 32.0)
            print('%s N=%5d L=%4d: %8.3f ms  -> %6.2f us per tile-step (tiles/dirs=%d, ~%.1f waves), %5.1f TFLOP/s' %
                  (name, N, L, ms, ms * 1e3 / (L * waves), tiles, waves, 2.0 * 4 * Hd * Hd * 2 * N * L / ms / 1e9), flush=True)
