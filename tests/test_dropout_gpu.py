"""Every dropout site of the library against the host reference of the counter RNG (tests/dropout_ref.py).

The masks are compared exactly, and the values bit for bit wherever the kernel only scales a copy: a failure names the
kernel whose index convention (or quad rule) has drifted from the one its forward / backward partner uses.
"""
import functools

import numpy as np
import pytest
import torch

from tests import dropout_ref as R
from tests.test_gemm_tc_gpu import EPI_PATHS

pytestmark = pytest.mark.gpu

SEEDS = [0, 0x2F3A5C7E9B1D4F61, 2 ** 62 - 1]
PS = [0.1, 0.25, 0.9]


def _ops():
    from nnr_b200 import ops
    return ops


@functools.lru_cache(maxsize=8)
def _grid_cpu(seed, rows, cols, p, ld=None):
    return torch.from_numpy(R.keep_scale_grid(seed, rows, cols, p, ld))


def _grid(seed, rows, cols, p, device, ld=None):
    """host keep-scale of a [rows, cols] block, element (r, c) at index r * ld + c, as a float32 tensor on ``device``"""
    return _grid_cpu(int(seed), rows, cols, float(p), ld).to(device)


def _randn_nz(*shape, generator):
    """N(0, 1) samples without exact zeros (a zero input would look dropped)"""
    x = torch.randn(*shape, generator=generator)
    x[x == 0] = 1.0
    return x


def _base(src):
    """value of a SeedSource's device base as the uint64 the kernels read"""
    return int(src.base.item()) & R.MASK64


def _seq(N, L, g, device):
    lens = torch.randint(1, L + 1, (N,), generator=g)
    len_ = lens.to(torch.int32).to(device)
    off = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(torch.int32).to(device)
    return lens, len_, off


def _slot_rows(lens, L):
    """padded slot index of every packed token (the counter the embedding masks use), in packed order"""
    return torch.cat([r * L + torch.arange(int(n)) for r, n in enumerate(lens.tolist())])


# ---------------------------------------------------------------------------------------------
# flat dropout
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('seed', SEEDS)
@pytest.mark.parametrize('p', PS)
def test_flat_dropout_matches_host_mask(cuda, seed, p):
    ops = _ops()
    g = torch.Generator().manual_seed(seed % 997 + int(100 * p))
    for n in (1, 4099, 10_000_003):
        x = _randn_nz(n, generator=g)
        s = torch.from_numpy(R.keep_scale(seed, np.arange(n, dtype=np.uint64), p))
        xd = x.to(cuda)
        y = torch.empty_like(xd)
        ops.dropout(xd, p, seed, y)
        y = y.cpu()
        assert torch.equal(y == 0, s == 0), (n, seed, p)
        assert torch.equal(y, x * s), (n, seed, p)                     # one fp32 product: bit exact
        ops.dropout(xd, p, seed, xd)                                   # in place (x is y)
        assert torch.equal(xd.cpu(), y), (n, seed, p)


# ---------------------------------------------------------------------------------------------
# embedding gather / scatter: counter = (r * L + t) * E + e, the padded slot
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('E', [300, 50])                  # float4 quads / scalar path (E % 4 != 0)
@pytest.mark.parametrize('seed', SEEDS)
@pytest.mark.parametrize('p', PS)
def test_embed_gather_matches_host_mask(cuda, E, seed, p):
    ops = _ops()
    g = torch.Generator().manual_seed(E + seed % 991 + int(100 * p))
    N, L, V = 53, 19, 97
    lens, len_, off = _seq(N, L, g, cuda)
    ntok = int(lens.sum())
    ids = torch.randint(0, V, (N, L), generator=g, dtype=torch.int32)
    table = _randn_nz(V, E, generator=g)
    slots = _slot_rows(lens, L)
    s_all = _grid(seed, N * L, E, p, 'cpu')
    s = s_all[slots]                                                   # [ntok, E] keep-scale of the packed rows
    tab_d, ids_d = table.to(cuda), ids.to(cuda)
    out_d = torch.full((N * L, E), float('nan'), device=cuda)
    ops.embed_gather_fwd(tab_d, ids_d, len_, off, out_d, p, seed)
    out = out_d[:ntok].cpu()
    rows = table[ids.view(-1).long()[slots]]
    assert torch.equal(out == 0, s == 0)
    assert torch.equal(out, rows * s)
    if E % 4:
        return                                                         # the scatter and the planes need E % 4 == 0
    # operand planes: same mask, same values as the fp32 gather split afterwards
    ref_pl = ops.tc_split(out_d, N * L, E, E, off[N:])
    if ref_pl is not None:                                             # None: the exact-fp32 GEMM backend has no planes
        pl = ops.embed_gather_planes_fwd(tab_d, ids_d, len_, off, N * L, p, seed)
        npl = ref_pl.buf.numel() // (N * L * ref_pl.pitch * ref_pl.esz)
        assert torch.equal(pl.buf.view(npl, N * L, -1)[:, :ntok], ref_pl.buf.view(npl, N * L, -1)[:, :ntok])
    # scatter: dtable = index_add(dout * mask)
    dout = torch.randn(N * L, E, generator=g)
    dtab = torch.empty(V, E, device=cuda)
    ops.embed_gather_bwd(dout.to(cuda), ids_d, len_, off, dtab, p, seed, False)
    ref = torch.zeros(V, E, dtype=torch.float64)
    ref.index_add_(0, ids.view(-1).long()[slots], dout[:ntok].double() * s.double())
    err = (dtab.cpu().double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 2e-6, (seed, p, err)


# ---------------------------------------------------------------------------------------------
# news vector: the category / sub-category embeddings, counter = r * (Ec + Es) + e, sub table at + Ec
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('modalities', [2, 1])             # 1: c_self = NULL (CNE_Title / CNE_Content)
@pytest.mark.parametrize('seed', SEEDS)
@pytest.mark.parametrize('p', PS)
def test_news_fuse_matches_host_mask(cuda, modalities, seed, p):
    ops = _ops()
    g = torch.Generator().manual_seed(modalities + seed % 983 + int(100 * p))
    N, D2, Ec, Es, nc, ns = 301, 40, 50, 30, 18, 41
    ts, tc, cs, cc = (torch.randn(N, D2, generator=g).to(cuda) for _ in range(4))
    if modalities == 1:
        cs = cc = None
    ct, st = _randn_nz(nc, Ec, generator=g).to(cuda), _randn_nz(ns, Es, generator=g).to(cuda)
    cat = torch.randint(0, nc, (N,), generator=g, dtype=torch.int32).to(cuda)
    sub = torch.randint(0, ns, (N,), generator=g, dtype=torch.int32).to(cuda)
    DM = modalities * D2
    s = _grid(seed, N, Ec + Es, p, cuda)
    out = torch.empty(N, DM + Ec + Es, device=cuda)
    ops.news_fuse_fwd(ts, tc, cs, cc, ct, st, cat, sub, N, D2, p, seed, out)
    parts = [ts + tc] + ([cs + cc] if modalities == 2 else [])
    ref = torch.cat(parts + [ct[cat.long()] * s[:, :Ec], st[sub.long()] * s[:, Ec:]], 1)
    assert torch.equal(out[:, DM:] == 0, s == 0)
    assert torch.equal(out, ref)
    dout = torch.randn(N, DM + Ec + Es, generator=g).to(cuda)
    d_a = torch.empty(N, D2, device=cuda)
    d_b = torch.empty(N, D2, device=cuda) if modalities == 2 else None
    dct, dst = torch.empty_like(ct), torch.empty_like(st)
    ops.news_fuse_bwd(dout, cat, sub, N, D2, p, seed, d_a, d_b, dct, dst, False)
    dm = dout.double()[:, DM:] * s.double()
    ref_c = torch.zeros(nc, Ec, dtype=torch.float64, device=cuda).index_add_(0, cat.long(), dm[:, :Ec])
    ref_s = torch.zeros(ns, Es, dtype=torch.float64, device=cuda).index_add_(0, sub.long(), dm[:, Ec:])
    for got, want in ((dct, ref_c), (dst, ref_s)):
        assert (got.double() - want).abs().max().item() < 1e-5 * want.abs().max().item(), (seed, p)
    dct2, dst2 = torch.empty_like(ct), torch.empty_like(st)
    ops.news_fuse_tables_bwd(dout, cat, sub, N, DM, p, seed, dct2, dst2, False)
    assert torch.equal(dct2, dct) and torch.equal(dst2, dst)


# ---------------------------------------------------------------------------------------------
# GEMM relu-residual epilogue: counter = m * N + n with the GEMM's N (not ldc)
# ---------------------------------------------------------------------------------------------
_GEMM_TOL = {'ALGO_AUTO': 4e-5, 'ALGO_BF16': 2e-2, 'ALGO_TF32X3': 2e-5, 'ALGO_SIMT': 1e-5}
_GEMM_CASES = ([('ALGO_AUTO', path) for path in EPI_PATHS] +
               [('ALGO_BF16', 'single'), ('ALGO_BF16', 'splitk4_m64'), ('ALGO_BF16', 'runtime_n225'),
                ('ALGO_TF32X3', 'single'), ('ALGO_TF32X3', 'pair'), ('ALGO_TF32X3', 'splitk_scalar'),
                ('ALGO_SIMT', 'single'), ('ALGO_SIMT', 'splitk_scalar')])


def _relu_res_gemm(ops, cuda, algo, path, p, seed, g):
    """runs EPI_BIAS_RELU_RES with aux = 1 + |N(0,1)| (so that a zero output means "dropped") on the path's shape and returns
    (out, aux_out, aux, z, Mv, N) with z = A B^T + bias in fp64, every tensor cut to the valid rows and the N columns"""
    c = EPI_PATHS[path]
    M, N, K, ldc = c['M'], c['N'], c['K'], c['ldc']
    Mv = c.get('m_dev', M)
    m_dev = torch.tensor([Mv], dtype=torch.int32, device=cuda) if 'm_dev' in c else None
    ld = c.get('ld', ldc)
    A = torch.randn(M, K, generator=g).to(cuda)
    W = (torch.randn(N, K, generator=g) / 40).to(cuda)
    bias = torch.randn(N, generator=g).to(cuda)
    aux = (1 + torch.randn(M, ld, generator=g).abs()).to(cuda)
    C = torch.full((M, ldc), float('nan'), device=cuda)
    ao = torch.full((M, ld), float('nan'), device=cuda)
    ops.gemm(A, W, C, M, N, K, K, K, ldc, False, True, ops.EPI_BIAS_RELU_RES, bias=bias, aux=aux, ldaux=ld, aux_out=ao,
             ldaux_out=ld, m_dev=m_dev, p_drop=p, seed=seed, algo=getattr(ops, algo))
    assert torch.isnan(C[:, N:]).all() and torch.isnan(C[Mv:]).all() and torch.isnan(ao[Mv:]).all()
    z = A[:Mv].double() @ W.double().t() + bias.double()
    return C[:Mv, :N], ao[:Mv, :N], aux[:Mv, :N], z, Mv, N


@pytest.mark.parametrize('algo,path', _GEMM_CASES)
def test_gemm_relu_res_epilogue_matches_host_mask(cuda, algo, path):
    ops = _ops()
    k = _GEMM_CASES.index((algo, path))
    seed, p = SEEDS[k % 3], PS[(k // 3) % 3]
    g = torch.Generator().manual_seed(100 + k)
    out, ao, aux, z, Mv, N = _relu_res_gemm(ops, cuda, algo, path, p, seed, g)
    s = _grid(seed, Mv, N, p, cuda)
    assert torch.equal(out == 0, s == 0), (algo, path)
    assert torch.equal(out, (ao + aux) * s), (algo, path)              # fp32(fp32(relu + aux) * scale), bit for bit
    r = torch.relu(z)
    assert (ao.double() - r).abs().max().item() < _GEMM_TOL[algo] * z.abs().max().item(), (algo, path)


@pytest.mark.parametrize('path', ['single', 'splitk4_m64', 'runtime_ld901'])
def test_gemm_relu_res_mask_matches_its_backward(cuda, path):
    """the backward recomputes the forward's mask: nnr_relu_bwd_split_colsum (dL/d pre-activation) and nnr_dropout on the
    [R, D] gradient of the residual branch, given the GEMM's seed, drop exactly the elements the GEMM dropped"""
    ops = _ops()
    if ops.default_algo() == ops.ALGO_SIMT:
        pytest.skip('planes exist only for the tensor-core GEMM algorithms')
    g = torch.Generator().manual_seed(7)
    seed, p = 0x2F3A5C7E9B1D4F61, 0.25
    out, ao, aux, z, R_, D = _relu_res_gemm(ops, cuda, 'ALGO_AUTO', path, p, seed, g)
    dropped = out == 0
    dy = (1 + torch.rand(R_, D, generator=g)).to(cuda)
    dd = torch.empty(R_, D, device=cuda)
    cs = torch.empty(D, device=cuda)
    ao_c = ao.contiguous()
    ops.relu_bwd_split_colsum(dy, ao_c, R_, D, p, seed, dd, cs)
    assert torch.equal(dd == 0, dropped)
    y = torch.empty_like(dy)
    ops.dropout(dy, p, seed, y)
    assert torch.equal(y == 0, dropped) and torch.equal(y, dd)


# ---------------------------------------------------------------------------------------------
# relu backward pre-pass: counter = r * C + c (C the column count, not the row stride)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('R_,C,ld', [(4352, 900, 900), (333, 50, 52), (130, 52, 56)])
@pytest.mark.parametrize('seed', SEEDS)
@pytest.mark.parametrize('p', PS)
def test_relu_backward_prepass_matches_host_mask(cuda, R_, C, ld, seed, p):
    ops = _ops()
    if ops.default_algo() == ops.ALGO_SIMT:
        pytest.skip('planes exist only for the tensor-core GEMM algorithms')
    g = torch.Generator().manual_seed(R_ + C + seed % 977 + int(100 * p))
    dy_full = torch.randn(R_, ld, generator=g).to(cuda)
    r_full = torch.relu(torch.randn(R_, ld, generator=g)).to(cuda)
    dy, r = dy_full[:, :C], r_full[:, :C]
    dd_full = torch.full((R_, ld), float('nan'), device=cuda)
    cs = torch.empty(C, device=cuda)
    pl = ops.relu_bwd_split_colsum(dy, r, R_, C, p, seed, dd_full[:, :C], cs)
    s = _grid(seed, R_, C, p, cuda)
    dd = dd_full[:, :C]
    assert torch.equal(dd == 0, (s == 0) | (dy == 0))
    assert torch.equal(dd, dy * s)
    assert torch.isnan(dd_full[:, C:]).all()
    dpre = dy * s * (r > 0)
    ref_pl = ops.tc_split(dpre.contiguous(), R_, C, C)
    assert torch.equal(pl.buf, ref_pl.buf)
    ref_cs = dpre.double().sum(0)
    assert (cs.double() - ref_cs).abs().max().item() < 1e-5 * max(1.0, ref_cs.abs().max().item())


# ---------------------------------------------------------------------------------------------
# indirect seeds: site k of a SeedSource resolves to mix64(base + k * golden) >> 2 in every kernel
# ---------------------------------------------------------------------------------------------
def test_indirect_seeds_resolve_like_the_host(cuda):
    ops = _ops()
    from nnr_b200 import engine
    torch.manual_seed(3)
    src = engine.SeedSource(cuda)
    base = _base(src)
    g = torch.Generator().manual_seed(11)
    p = 0.25

    def host(seed):
        return R.resolve_seed(seed, base)

    # nnr_dropout
    sd = src.next()
    n = 100_003
    x = torch.randn(n, generator=g).to(cuda)
    y = torch.empty_like(x)
    ops.dropout(x, p, sd, y)
    assert torch.equal(y, x * torch.from_numpy(R.keep_scale(host(sd), np.arange(n, dtype=np.uint64), p)).to(cuda))
    # the GEMM epilogue, compile-time path and split-K path
    for path in ('single', 'splitk4_m64'):
        sd = src.next()
        out, ao, aux, z, Mv, N = _relu_res_gemm(ops, cuda, 'ALGO_AUTO', path, p, sd, g)
        assert torch.equal(out, (ao + aux) * _grid(host(sd), Mv, N, p, cuda)), path
    # embedding gather / scatter
    sd = src.next()
    N, L, V, E = 41, 13, 57, 300
    lens, len_, off = _seq(N, L, g, cuda)
    ntok = int(lens.sum())
    ids = torch.randint(0, V, (N, L), generator=g, dtype=torch.int32)
    table = torch.randn(V, E, generator=g)
    slots = _slot_rows(lens, L)
    s = _grid(host(sd), N * L, E, p, 'cpu')[slots]
    out = torch.empty(N * L, E, device=cuda)
    ops.embed_gather_fwd(table.to(cuda), ids.to(cuda), len_, off, out, p, sd)
    assert torch.equal(out[:ntok].cpu(), table[ids.view(-1).long()[slots]] * s)
    dout = torch.randn(N * L, E, generator=g)
    dtab = torch.empty(V, E, device=cuda)
    ops.embed_gather_bwd(dout.to(cuda), ids.to(cuda), len_, off, dtab, p, sd, False)
    ref = torch.zeros(V, E, dtype=torch.float64).index_add_(0, ids.view(-1).long()[slots], dout[:ntok].double() * s.double())
    assert (dtab.cpu().double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()
    # news vector forward and table gradients
    sd = src.next()
    Nn, D2, Ec, Es, nc, ns = 97, 16, 50, 30, 9, 13
    ts = torch.randn(Nn, D2, generator=g).to(cuda)
    ct, st = torch.randn(nc, Ec, generator=g).to(cuda), torch.randn(ns, Es, generator=g).to(cuda)
    cat = torch.randint(0, nc, (Nn,), generator=g, dtype=torch.int32).to(cuda)
    sub = torch.randint(0, ns, (Nn,), generator=g, dtype=torch.int32).to(cuda)
    s = _grid(host(sd), Nn, Ec + Es, p, cuda)
    o = torch.empty(Nn, D2 + Ec + Es, device=cuda)
    ops.news_fuse_fwd(ts, None, None, None, ct, st, cat, sub, Nn, D2, p, sd, o)
    assert torch.equal(o, torch.cat([ts, ct[cat.long()] * s[:, :Ec], st[sub.long()] * s[:, Ec:]], 1))
    do = torch.randn(Nn, D2 + Ec + Es, generator=g).to(cuda)
    dct, dst = torch.empty_like(ct), torch.empty_like(st)
    ops.news_fuse_tables_bwd(do, cat, sub, Nn, D2, p, sd, dct, dst, False)
    dm = do.double()[:, D2:] * s.double()
    ref_c = torch.zeros(nc, Ec, dtype=torch.float64, device=cuda).index_add_(0, cat.long(), dm[:, :Ec])
    ref_s = torch.zeros(ns, Es, dtype=torch.float64, device=cuda).index_add_(0, sub.long(), dm[:, Ec:])
    assert (dct.double() - ref_c).abs().max().item() < 1e-5 * ref_c.abs().max().item()
    assert (dst.double() - ref_s).abs().max().item() < 1e-5 * ref_s.abs().max().item()
    # layer norm + relu + residual, forward and backward
    sd = src.next()
    Rl, D = 301, 900
    yv = torch.randn(Rl, D, generator=g).to(cuda)
    res = (1 + torch.randn(Rl, D, generator=g).abs()).to(cuda)
    gamma, beta = torch.ones(D, device=cuda), torch.zeros(D, device=cuda)
    lo, rl = torch.empty(Rl, D, device=cuda), torch.empty(Rl, D, device=cuda)
    mu, rstd = torch.empty(Rl, device=cuda), torch.empty(Rl, device=cuda)
    ops.ln_relu_res_fwd(yv, gamma, beta, res, Rl, D, 1e-5, p, sd, lo, rl, mu, rstd)
    s = _grid(host(sd), Rl, D, p, cuda)
    assert torch.equal(lo == 0, s == 0) and torch.equal(lo, (rl + res) * s)
    dl = torch.randn(Rl, D, generator=g).to(cuda)
    dd = torch.empty(Rl, D, device=cuda)
    dyl, dgam, dbet = torch.empty(Rl, D, device=cuda), torch.empty(D, device=cuda), torch.empty(D, device=cuda)
    ops.ln_relu_res_bwd(dl, yv, gamma, rl, mu, rstd, Rl, D, p, sd, dd, dyl, dgam, dbet)
    assert torch.equal(dd, dl * s)


def test_forward_and_backward_partners_share_the_indirect_mask(cuda):
    """given the same indirect seed, the news vector's forward and its table backward drop the same elements, and so do
    the GEMM epilogue and the backward pre-pass / nnr_dropout that recompute its mask"""
    ops = _ops()
    from nnr_b200 import engine
    src = engine.SeedSource(cuda)
    g = torch.Generator().manual_seed(12)
    p = 0.25
    sd = src.next()
    N, D2, Ec, Es, nc, ns = 200, 8, 50, 30, 200, 200
    ct, st = torch.ones(nc, Ec, device=cuda), torch.ones(ns, Es, device=cuda)
    ar = torch.arange(N, dtype=torch.int32, device=cuda)               # row r takes table row r: dtable = dout * mask
    o = torch.empty(N, D2 + Ec + Es, device=cuda)
    ops.news_fuse_fwd(torch.zeros(N, D2, device=cuda), None, None, None, ct, st, ar, ar, N, D2, p, sd, o)
    dct, dst = torch.empty_like(ct), torch.empty_like(st)
    ops.news_fuse_tables_bwd(torch.ones_like(o), ar, ar, N, D2, p, sd, dct, dst, False)
    assert torch.equal(torch.cat([dct, dst], 1), o[:, D2:])
    if ops.default_algo() == ops.ALGO_SIMT:
        return
    sd = src.next()
    out, ao, aux, z, R_, D = _relu_res_gemm(ops, cuda, 'ALGO_AUTO', 'single', p, sd, g)
    dy = torch.ones(R_, D, device=cuda)
    dd, cs = torch.empty(R_, D, device=cuda), torch.empty(D, device=cuda)
    ops.relu_bwd_split_colsum(dy, ao.contiguous(), R_, D, p, sd, dd, cs)
    y = torch.empty_like(dy)
    ops.dropout(dy, p, sd, y)
    assert torch.equal(dd == 0, out == 0) and torch.equal(y, dd)


def test_graph_replays_draw_the_mask_of_the_current_base(cuda):
    """nnr_dropout and a compile-time-epilogue GEMM captured in a CUDA graph with indirect seeds: after advance() every
    replay draws the host mask of the new base, and no two replays are alike"""
    ops = _ops()
    from nnr_b200 import engine
    src = engine.SeedSource(cuda)
    g = torch.Generator().manual_seed(13)
    p = 0.25
    n = 1 << 16
    x = torch.randn(n, generator=g).to(cuda)
    y = torch.empty_like(x)
    M, N, K = 4352, 900, 900                                            # EPI_PATHS['single']: compile-time epilogue
    A = torch.randn(M, K, generator=g).to(cuda)
    W = (torch.randn(N, K, generator=g) / 40).to(cuda)
    bias = torch.randn(N, generator=g).to(cuda)
    aux = (1 + torch.randn(M, N, generator=g).abs()).to(cuda)
    C, ao = torch.empty(M, N, device=cuda), torch.empty(M, N, device=cuda)
    s_drop, s_gemm = src.next(), src.next()

    def step():
        ops.dropout(x, p, s_drop, y)
        ops.gemm(A, W, C, M, N, K, K, K, N, False, True, ops.EPI_BIAS_RELU_RES, bias=bias, aux=aux, ldaux=N, aux_out=ao,
                 ldaux_out=N, p_drop=p, seed=s_gemm)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()                                                          # warm-up: workspaces exist before the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    seen = []
    for _ in range(3):
        src.advance()
        graph.replay()
        torch.cuda.synchronize()
        base = _base(src)
        sx = torch.from_numpy(R.keep_scale(R.resolve_seed(s_drop, base), np.arange(n, dtype=np.uint64), p)).to(cuda)
        assert torch.equal(y, x * sx)
        sg = _grid(R.resolve_seed(s_gemm, base), M, N, p, cuda)
        assert torch.equal(C, (ao + aux) * sg)
        seen.append((y.clone(), C.clone()))
    for i in range(3):
        for j in range(i):
            assert not torch.equal(seen[i][0], seen[j][0]) and not torch.equal(seen[i][1], seen[j][1])
