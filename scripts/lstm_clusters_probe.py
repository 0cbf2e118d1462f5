import sys
sys.path.insert(0, '/root/repo')
import ctypes, torch
from nnr_b200 import ops
from nnr_b200._lib import lib
dev = torch.device('cuda:0'); Hd = 200; N, L = 3520, 16
lens = torch.full((N,), L, dtype=torch.int32, device=dev)
off = (torch.arange(N + 1, device=dev) * L).to(torch.int32)
order = torch.arange(N, dtype=torch.int32, device=dev)
gx = torch.randn(N * L, 8 * Hd, device=dev) * 0.1
w_hh = torch.randn(2, 4 * Hd, Hd, device=dev) * 0.05
h = torch.empty(N * L, 2 * Hd, device=dev); cst = torch.empty(N * L, 2 * Hd, device=dev); cn = torch.empty(N, 2 * Hd, device=dev)
ops.lstm_fwd(gx, w_hh, lens, off, order, N, L, Hd, h, cst, cn); torch.cuda.synchronize()
lib.nnr_debug_lstm_clusters.restype = ctypes.c_int
print('max active clusters:', lib.nnr_debug_lstm_clusters())
