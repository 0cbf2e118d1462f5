"""Small invocations of the kernels that use clusters / mbarriers / DSMEM / TMA, sized for compute-sanitizer
(racecheck and synccheck slow a kernel down by two orders of magnitude):

    compute-sanitizer --tool racecheck python scripts/sanitize_targets.py lstm
    compute-sanitizer --tool synccheck python scripts/sanitize_targets.py gemm
    compute-sanitizer --tool memcheck  python scripts/sanitize_targets.py embed

targets: lstm (lstm_fwd_tm_kernel / lstm_bwd_mma_kernel, 5-CTA clusters, bulk-copy exchange), gemm (gemm_tc_kernel<1,0> and the
CTA-pair gemm_tc_kernel<1,1>, TMA + tcgen05 + mbarriers), embed (eb_keys / radix sort / eb_chunk / eb_fix scatter)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from nnr_b200 import ops  # noqa: E402

dev = torch.device('cuda:0')
what = sys.argv[1] if len(sys.argv) > 1 else 'lstm'
torch.manual_seed(0)

if what == 'lstm':
    N, L, Hd = 70, 9, 200
    lens = torch.randint(1, L + 1, (N,))
    lens[0] = L
    off = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(torch.int32).to(dev)
    len_ = lens.to(torch.int32).to(dev)
    order = torch.sort(lens, descending=True, stable=True)[1].to(torch.int32).to(dev)
    gx = torch.randn(N * L, 8 * Hd, device=dev) * 0.3
    w_hh = torch.randn(2, 4 * Hd, Hd, device=dev) * 0.07
    h = torch.zeros(N * L, 2 * Hd, device=dev)
    cst = torch.zeros(N * L, 2 * Hd, device=dev)
    cn = torch.zeros(N, 2 * Hd, device=dev)
    ops.lstm_fwd(gx, w_hh, len_, off, order, N, L, Hd, h, cst, cn)
    dh = torch.randn(N * L, 2 * Hd, device=dev) * 0.1
    dcn = torch.randn(N, 2 * Hd, device=dev) * 0.1
    db = torch.empty(8 * Hd, device=dev)
    ops.lstm_bwd_planes(gx, cst, w_hh, len_, off, order, N, L, Hd, dh, dcn, N * L, db)
    ops.lstm_bwd(gx, cst, w_hh, len_, off, order, N, L, Hd, dh, dcn)
    torch.cuda.synchronize()
    print('lstm ok', float(h.abs().sum()), float(gx.abs().sum()))
elif what == 'gemm':
    for (M, N, K, tA, tB, epi) in [(300, 200, 400, False, True, ops.EPI_BIAS_TANH), (400, 400, 1500, True, False, ops.EPI_NONE),
                                   (2 * 128 * 148 + 300, 96, 64, False, True, ops.EPI_NONE)]:      # the last one: CTA pairs
        A = torch.randn((K, M) if tA else (M, K), device=dev)
        B = torch.randn((N, K) if tB else (K, N), device=dev)
        C = torch.empty(M, N, device=dev)
        bias = torch.randn(N, device=dev)
        ops.gemm(A, B, C, M, N, K, A.stride(0), B.stride(0), N, tA, tB, epi, bias=bias if epi else None)
        torch.cuda.synchronize()
        ref = (A.t() if tA else A).double() @ (B.t() if tB else B).double()
        if epi == ops.EPI_BIAS_TANH:
            ref = torch.tanh(ref + bias.double())
        print('gemm', M, N, K, 'max err', float((C.double() - ref).abs().max()))
elif what == 'embed':
    N, L, E, V = 40, 12, 300, 57
    lens = torch.randint(1, L + 1, (N,))
    off = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(torch.int32).to(dev)
    len_ = lens.to(torch.int32).to(dev)
    ids = torch.randint(0, V, (N, L), dtype=torch.int32, device=dev)
    dout = torch.randn(N * L, E, device=dev)
    dtable = torch.zeros(V, E, device=dev)
    ops.embed_gather_bwd(dout, ids, len_, off, dtable, 0.2, 77, False)
    ops.embed_gather_bwd(dout, ids, len_, off, dtable, 0.0, 0, True)
    torch.cuda.synchronize()
    print('embed ok', float(dtable.abs().sum()))
