"""The per-news / SUE-sized GEMMs (a few thousand rows) in isolation: CUDA-event time per call at three contraction lengths,
from which the fixed cost of a launch (prologue + the last tile's epilogue) and the cost per 64-deep k-block separate.

    python scripts/gemm_sue_probe.py [reps]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from nnr_b200 import ops  # noqa: E402
from nnr_b200.ops import EPI_BIAS, EPI_BIAS_RELU_RES, EPI_NONE  # noqa: E402

dev = torch.device('cuda:0')
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 20
torch.manual_seed(0)


def timed(fn):
    fn(); fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / REPS * 1e3


for (M, N, tB, epi) in ((4352, 900, True, EPI_NONE), (4352, 900, True, EPI_BIAS_RELU_RES), (4352, 900, False, EPI_NONE),
                        (3520, 400, True, EPI_BIAS), (6080, 900, True, EPI_NONE)):
    row = []
    for K in (64, 896, 1792):
        x = torch.randn(M, K, device=dev)
        W = torch.randn((N, K) if tB else (K, N), device=dev) * 0.05
        out = torch.empty(M, N, device=dev)
        aux = torch.randn(M, N, device=dev)
        aux_out = torch.empty(M, N, device=dev)
        bias = torch.randn(N, device=dev)
        x_pl = ops.tc_split(x, M, K, K)
        w_pl = ops.tc_split(W, W.shape[0], W.shape[1], W.shape[1])
        kw = {}
        if epi == EPI_BIAS_RELU_RES:
            kw = dict(bias=bias, aux=aux, ldaux=N, aux_out=aux_out, ldaux_out=N, p_drop=0.2, seed=1234)
        elif epi == EPI_BIAS:
            kw = dict(bias=bias)

        def fn():
            ops.gemm(x, W, out, M, N, K, K, W.stride(0), N, False, tB, epi, a_planes=x_pl, b_planes=w_pl, **kw)
        row.append(timed(fn))
    per_kb = (row[2] - row[1]) / 14.0
    print('%5dx%4d %s e%d: K=64 %6.1f us   K=896 %6.1f us   K=1792 %6.1f us   -> %5.2f us per k-block, fixed ~%5.1f us' %
          (M, N, 'NT' if tB else 'NN', epi, row[0], row[1], row[2], per_kb, row[1] - 14 * per_kb), flush=True)
