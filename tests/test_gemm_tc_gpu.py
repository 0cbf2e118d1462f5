"""GPU tests of the tcgen05 (3xTF32 / BF16) GEMM backend against fp64 torch and the exact-fp32 FFMA backend."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

# max|err| / max|ref|.  The hi/lo split itself is good to ~2^-21, but the tensor core adds the products of one
# tcgen05.mma into the fp32 TMEM accumulator with truncation, which leaves ~2^-24 x (MMAs in the chain) of bias:
# measured 4e-6 at K=400, 1.1e-5 at K=1600.  nnr_gemm bounds the chain with split-K (<= 1024 k per partial sum).
TF32X3_TOL = 2e-5
BF16_TOL = 2e-2


def _ref(A, B, transA, transB):
    a = A.double().t() if transA else A.double()
    b = B.double().t() if transB else B.double()
    return a @ b


def _run(ops, A, B, M, N, K, transA, transB, algo, **kw):
    C = torch.full((M, N), float('nan'), device=A.device)
    ops.gemm(A, B, C, M, N, K, A.stride(0), B.stride(0), N, transA, transB, algo=algo, **kw)
    return C


@pytest.mark.parametrize('shape', [(1000, 1600, 300), (513, 400, 400), (260, 200, 225), (256, 256, 64), (3000, 300, 1600),
                                   (640, 900, 900), (777, 225, 900)])
def test_tf32x3_all_layouts(cuda, shape):
    from nnr_b200 import ops
    M, N, K = shape
    g = torch.Generator().manual_seed(M + N + K)
    for transA in (False, True):
        for transB in (False, True):
            A = torch.randn((K, M) if transA else (M, K), generator=g).to(cuda)
            B = torch.randn((N, K) if transB else (K, N), generator=g).to(cuda)
            C = _run(ops, A, B, M, N, K, transA, transB, ops.ALGO_TF32X3)
            ref = _ref(A, B, transA, transB)
            err = (C.double() - ref).abs().max().item() / ref.abs().max().item()
            assert err < TF32X3_TOL, (shape, transA, transB, err)


def test_tf32x3_wide_dynamic_range(cuda):
    """hi/lo split must hold when operand magnitudes span many binades"""
    from nnr_b200 import ops
    g = torch.Generator().manual_seed(5)
    M, N, K = 512, 400, 400
    A = (torch.randn(M, K, generator=g) * torch.exp(torch.randn(M, K, generator=g) * 3)).to(cuda)
    B = (torch.randn(N, K, generator=g) * torch.exp(torch.randn(N, K, generator=g) * 3)).to(cuda)
    C = _run(ops, A, B, M, N, K, False, True, ops.ALGO_TF32X3)
    ref = A.double() @ B.double().t()
    scale = (A.double().abs() @ B.double().abs().t())
    assert ((C.double() - ref).abs() / scale).max().item() < 2e-5


def test_tf32x3_device_bounds_and_splitk(cuda):
    from nnr_b200 import ops
    g = torch.Generator().manual_seed(6)
    M, N, K = 40000, 300, 1600            # wgrad: out[1600,300] = dy^T x, contraction over 40000 tokens
    dy = torch.randn(M, K, generator=g).to(cuda)
    x = torch.randn(M, N, generator=g).to(cuda)
    for kd in (M, 12345, 33, 1):
        k_dev = torch.tensor([kd], dtype=torch.int32, device=cuda)
        out = torch.full((K, N), float('nan'), device=cuda)
        ops.gemm(dy, x, out, K, N, M, K, N, N, True, False, k_dev=k_dev, algo=ops.ALGO_TF32X3)
        ref = dy[:kd].double().t() @ x[:kd].double()
        err = (out.double() - ref).abs().max().item() / ref.abs().max().item()
        assert err < TF32X3_TOL, (kd, err)
        out2 = torch.empty_like(out)
        ops.gemm(dy, x, out2, K, N, M, K, N, N, True, False, k_dev=k_dev, algo=ops.ALGO_TF32X3)
        assert torch.equal(out, out2)
    # m_dev: rows beyond *m_dev untouched; garbage (NaN) rows beyond m_dev in A must not leak
    W = torch.randn(200, N, generator=g).to(cuda)
    xa = x.clone()
    xa[777:] = float('nan')
    out = torch.full((M, 200), 7.0, device=cuda)
    m_dev = torch.tensor([777], dtype=torch.int32, device=cuda)
    ops.gemm(xa, W, out, M, 200, N, N, N, 200, False, True, m_dev=m_dev, algo=ops.ALGO_TF32X3)
    ref = x[:777].double() @ W.double().t()
    assert (out[:777].double() - ref).abs().max().item() / ref.abs().max().item() < TF32X3_TOL
    assert torch.all(out[777:] == 7.0)


def test_tf32x3_epilogues_match_ffma_backend(cuda):
    from nnr_b200 import ops
    g = torch.Generator().manual_seed(7)
    M, N, K = 1333, 400, 400
    A = torch.randn(M, K, generator=g).to(cuda)
    W = (torch.randn(N, K, generator=g) / 20).to(cuda)
    bias = torch.randn(N, generator=g).to(cuda)
    aux = torch.randn(M, N, generator=g).to(cuda)
    rowmap = torch.randint(0, 10, (M,), generator=g, dtype=torch.int32).to(cuda)
    rowbias = torch.randn(10, N, generator=g).to(cuda)
    cases = [dict(epilogue=ops.EPI_BIAS, bias=bias), dict(epilogue=ops.EPI_BIAS_TANH, bias=bias),
             dict(epilogue=ops.EPI_BIAS_RELU_RES, bias=bias, aux=aux, ldaux=N, p_drop=0.25, seed=5),
             dict(epilogue=ops.EPI_GATE, rowbias=rowbias, ldrowbias=N, rowmap=rowmap, aux=aux, ldaux=N),
             dict(epilogue=ops.EPI_ADD_AUX, aux=aux, ldaux=N)]
    for kw in cases:
        outs = []
        for algo in (ops.ALGO_SIMT, ops.ALGO_TF32X3):
            aux_out = torch.zeros(M, N, device=cuda)
            extra = dict(aux_out=aux_out, ldaux_out=N) if kw['epilogue'] in (ops.EPI_BIAS_RELU_RES, ops.EPI_GATE) else {}
            outs.append((_run(ops, A, W, M, N, K, False, True, algo, **kw, **extra), aux_out))
        assert (outs[0][0] - outs[1][0]).abs().max().item() < 1e-4, kw['epilogue']
        assert (outs[0][1] - outs[1][1]).abs().max().item() < 1e-4, kw['epilogue']
    base = torch.randn(M, N, generator=g).to(cuda)
    o1, o2 = base.clone(), base.clone()
    ops.gemm(A, W, o1, M, N, K, K, K, N, False, True, accumulate=True, algo=ops.ALGO_SIMT)
    ops.gemm(A, W, o2, M, N, K, K, K, N, False, True, accumulate=True, algo=ops.ALGO_TF32X3)
    assert (o1 - o2).abs().max().item() < 1e-4


def test_bf16_variant(cuda):
    from nnr_b200 import ops
    g = torch.Generator().manual_seed(8)
    for (M, N, K) in [(1000, 1600, 300), (513, 400, 400), (3000, 300, 1600)]:
        for transA, transB in ((False, True), (False, False), (True, False)):
            A = torch.randn((K, M) if transA else (M, K), generator=g).to(cuda)
            B = torch.randn((N, K) if transB else (K, N), generator=g).to(cuda)
            C = _run(ops, A, B, M, N, K, transA, transB, ops.ALGO_BF16)
            ref = _ref(A, B, transA, transB)
            err = (C.double() - ref).abs().max().item() / ref.abs().max().item()
            assert err < BF16_TOL, (M, N, K, transA, transB, err)
            # exact against a bf16-rounded fp32 product
            a = (A.t() if transA else A).bfloat16().double()
            b = (B.t() if transB else B).bfloat16().double()
            err2 = (C.double() - a @ b).abs().max().item() / ref.abs().max().item()
            assert err2 < 1e-5, (M, N, K, err2)


def test_bf16x3_variant(cuda):
    """bf16 hi/lo split (3 MMAs of kind::f16): operands carry 16 mantissa bits -> ~1e-5 of max|C|"""
    from nnr_b200 import ops
    g = torch.Generator().manual_seed(9)
    worst = 0.0
    for (M, N, K) in [(1000, 1600, 300), (513, 400, 400), (3000, 300, 1600), (777, 225, 900)]:
        for transA, transB in ((False, True), (False, False), (True, False), (True, True)):
            A = torch.randn((K, M) if transA else (M, K), generator=g).to(cuda)
            B = torch.randn((N, K) if transB else (K, N), generator=g).to(cuda)
            C = _run(ops, A, B, M, N, K, transA, transB, ops.ALGO_BF16X3)
            ref = _ref(A, B, transA, transB)
            err = (C.double() - ref).abs().max().item() / ref.abs().max().item()
            worst = max(worst, err)
            assert err < 4e-5, (M, N, K, transA, transB, err)
    print('bf16x3 worst rel err', worst)


@pytest.mark.parametrize('algo_name', ['ALGO_BF16X3', 'ALGO_TF32X3'])
def test_cta_pair_tiles_large_m(cuda, algo_name):
    """Row counts >= 2*128*148 run on CTA pairs (cta_group::2, 256-row tiles, B tile split across the pair):
    device-side row bound, N tails, every epilogue input, both B layouts that qualify."""
    from nnr_b200 import ops
    algo = getattr(ops, algo_name)
    g = torch.Generator().manual_seed(17)
    cap, Mv = 40000, 38211                                     # capacity and device-side valid rows (odd tail)
    m_dev = torch.tensor([Mv], dtype=torch.int32, device=cuda)
    for (N, K, transB) in [(1600, 300, True), (400, 400, True), (200, 400, True), (300, 96, True), (256, 200, False)]:
        A = torch.randn(cap, K, generator=g).to(cuda)
        B = torch.randn((N, K) if transB else (K, N), generator=g).to(cuda)
        bias = torch.randn(N, generator=g).to(cuda)
        C = torch.full((cap, N), float('nan'), device=cuda)
        ops.gemm(A, B, C, cap, N, K, A.stride(0), B.stride(0), N, False, transB, ops.EPI_BIAS, bias=bias, m_dev=m_dev, algo=algo)
        ref = A[:Mv].double() @ (B.double().t() if transB else B.double()) + bias.double()
        err = (C[:Mv].double() - ref).abs().max().item() / ref.abs().max().item()
        assert err < 4e-5, (N, K, transB, err)
        assert torch.isnan(C[Mv:]).all()                       # rows beyond the device bound are not written
    # gate epilogue (row bias through a row map, aux in, aux out) on the pair path
    N, K = 400, 400
    A = torch.randn(cap, K, generator=g).to(cuda)
    W = torch.randn(N, K, generator=g).to(cuda) * 0.05
    rb = torch.randn(77, N, generator=g).to(cuda)
    rmap = torch.randint(0, 77, (cap,), generator=g).to(torch.int32).to(cuda)
    gate = torch.empty(cap, N, device=cuda)
    C = torch.empty(cap, N, device=cuda)
    ops.gemm(A, W, C, cap, N, K, K, K, N, False, True, ops.EPI_GATE, rowbias=rb, ldrowbias=N, rowmap=rmap, aux=A, ldaux=K,
             aux_out=gate, ldaux_out=N, m_dev=m_dev, algo=algo)
    gref = torch.sigmoid(A[:Mv].double() @ W.double().t() + rb.double()[rmap[:Mv].long()])
    assert (gate[:Mv].double() - gref).abs().max().item() < 2e-5
    assert (C[:Mv].double() - gref * A[:Mv].double()).abs().max().item() < 1e-4


# The kernel paths that finish a default-algorithm (bf16x3) GEMM's epilogue, each with an NT shape that make_plan
# (gemm_tc.cu) sends there.  ldc > N where the path allows it, so a column index taken from ldc instead of N shows.
EPI_PATHS = {
    # N % 4 == 0, 16-byte aligned operands, 34 x 7 = 238 tiles (more than 74: no split-K): the compile-time epilogue of the
    # single-CTA kernel; block_n 144 leaves a 36-column N tail
    'single': dict(M=4352, N=900, K=900, ldc=904),
    # M >= 2 * 128 * 148 = 37 888, A row-major, no k_dev: 256-row tiles on CTA pairs (compile-time epilogue); the device-side
    # row count ends inside a tile
    'pair': dict(M=40000, N=900, K=900, ldc=904, m_dev=38211),
    # tiles * 2 <= 148 and ceil(K / 64) = 15 >= 8: split-K partials, combined with the epilogue by tc_splitk_reduce4_kernel
    # (N % 4 == 0)
    'splitk4_m64': dict(M=64, N=900, K=900, ldc=904, splits=4),
    'splitk4_m640': dict(M=640, N=900, K=900, ldc=904, splits=4),
    # split-K with N % 4 != 0: the scalar tc_splitk_reduce_kernel
    'splitk_scalar': dict(M=320, N=225, K=900, ldc=225, splits=4),
    # N % 4 != 0 and 79 x 2 = 158 tiles (no split): the run-time-switched epilogue
    'runtime_n225': dict(M=10000, N=225, K=900, ldc=225),
    # leading dimensions of 901 floats (rows not 16-byte aligned): the run-time-switched epilogue at N % 4 == 0
    'runtime_ld901': dict(M=4352, N=900, K=900, ldc=901, ld=901),
}


def _gemm_workspace_bytes(A, B, C, M, N, K, ldc):
    from nnr_b200 import _lib, ops
    a = _lib.GemmArgs()
    a.A, a.lda, a.B, a.ldb, a.transB, a.C, a.ldc = A.data_ptr(), K, B.data_ptr(), K, 1, C.data_ptr(), ldc
    a.M, a.N, a.K, a.algo = M, N, K, ops.ALGO_AUTO
    return int(_lib.lib.nnr_gemm_workspace_bytes(ctypes.byref(a)))


@pytest.mark.parametrize('path', list(EPI_PATHS))
def test_default_epilogues_on_each_kernel_path(cuda, path):
    """every epilogue of the default algorithm against fp64 on each kernel path that can finish it: values, rows >= m_dev
    and columns [N, ldc) left untouched, and a repeated call bit-identical"""
    from nnr_b200 import ops
    from tests import dropout_ref
    if ops.default_algo() != ops.ALGO_BF16X3:
        pytest.skip('paths and tolerances of the bf16x3 default')
    c = EPI_PATHS[path]
    M, N, K, ldc = c['M'], c['N'], c['K'], c['ldc']
    ld = c.get('ld', ldc)
    Mv = c.get('m_dev', M)
    m_dev = torch.tensor([Mv], dtype=torch.int32, device=cuda) if 'm_dev' in c else None
    g = torch.Generator().manual_seed(M + N + ldc)
    A = torch.randn(M, K, generator=g).to(cuda)
    W = (torch.randn(N, K, generator=g) / 80).to(cuda)          # |A W^T| ~ 0.4: tanh / sigmoid are not saturated
    bias = torch.randn(N, generator=g).to(cuda)
    aux = torch.randn(M, ld, generator=g).to(cuda)
    rowmap = torch.randint(0, 37, (M,), generator=g, dtype=torch.int32).to(cuda)
    rowbias = torch.randn(37, ld, generator=g).to(cuda)
    base = torch.randn(M, ldc, generator=g).to(cuda)
    if 'splits' in c:                                          # the partial sums really are split: [splits][M][N] fp32
        C0 = torch.empty(M, ldc, device=cuda)
        planes = sum((rows * ((K + 7) // 8 * 8) * 4 + 1023) // 1024 * 1024 for rows in (M, N))
        assert _gemm_workspace_bytes(A, W, C0, M, N, K, ldc) - planes == (c['splits'] * M * N * 4 + 1023) // 1024 * 1024
    prod = A[:Mv].double() @ W.double().t()
    z = prod + bias.double()
    zmax = z.abs().max().item()
    ax = aux[:Mv, :N].double()
    s = torch.from_numpy(dropout_ref.keep_scale_grid(77, Mv, N, 0.25)).to(cuda).double()
    rb = rowbias.double()[rowmap[:Mv].long(), :N]
    sig = torch.sigmoid(prod + rb)
    # (name, kwargs, fp64 reference of C, absolute tolerance of C, reference of aux_out or None)
    cases = [('bias', dict(epilogue=ops.EPI_BIAS, bias=bias), z, 4e-5 * zmax, None),
             ('bias_tanh', dict(epilogue=ops.EPI_BIAS_TANH, bias=bias), torch.tanh(z), 2e-5, None),
             ('relu', dict(epilogue=ops.EPI_BIAS_RELU_RES, bias=bias), torch.relu(z), 4e-5 * zmax, None),
             ('relu_res', dict(epilogue=ops.EPI_BIAS_RELU_RES, bias=bias, aux=aux, ldaux=ld), torch.relu(z) + ax,
              4e-5 * zmax, torch.relu(z)),
             ('relu_res_drop', dict(epilogue=ops.EPI_BIAS_RELU_RES, bias=bias, aux=aux, ldaux=ld, p_drop=0.25, seed=77),
              (torch.relu(z) + ax) * s, 4e-5 * zmax * 4 / 3, torch.relu(z)),
             ('gate', dict(epilogue=ops.EPI_GATE, rowbias=rowbias, ldrowbias=ld, rowmap=rowmap, aux=aux, ldaux=ld), sig * ax,
              2e-5 * ax.abs().max().item(), sig),
             ('add_aux', dict(epilogue=ops.EPI_ADD_AUX, aux=aux, ldaux=ld), prod + ax, 4e-5 * zmax, None),
             ('accumulate', dict(epilogue=ops.EPI_NONE, accumulate=True), prod + base[:Mv, :N].double(), 4e-5 * zmax, None)]
    for name, kw, ref, tol, ao_ref in cases:
        outs = []
        for _ in range(2):
            C = base.clone() if kw.get('accumulate') else torch.full((M, ldc), float('nan'), device=cuda)
            ao = torch.full((M, ld), float('nan'), device=cuda) if ao_ref is not None else None
            extra = dict(aux_out=ao, ldaux_out=ld) if ao is not None else {}
            ops.gemm(A, W, C, M, N, K, K, K, ldc, False, True, m_dev=m_dev, **kw, **extra)
            outs.append((C, ao))
        C, ao = outs[0]
        err = (C[:Mv, :N].double() - ref).abs().max().item()
        assert err < tol, (path, name, err, tol)
        if kw.get('accumulate'):
            assert torch.equal(C[Mv:], base[Mv:]) and torch.equal(C[:, N:], base[:, N:]), (path, name)
        else:
            assert torch.isnan(C[Mv:]).all() and torch.isnan(C[:, N:]).all(), (path, name)
        assert torch.equal(outs[1][0][:Mv, :N], C[:Mv, :N]), (path, name)
        if ao_ref is not None:
            err = (ao[:Mv, :N].double() - ao_ref).abs().max().item()
            assert err < (2e-5 if name == 'gate' else 4e-5 * zmax), (path, name, err)
            assert torch.isnan(ao[Mv:]).all() and torch.isnan(ao[:, N:]).all(), (path, name)
            assert torch.equal(outs[1][1][:Mv, :N], ao[:Mv, :N]), (path, name)


@pytest.mark.parametrize('cols', [1600, 200, 300, 96])
def test_split_with_column_sums(cuda, cols):
    """nnr_tc_split_colsum: same planes as nnr_tc_split (bit-exact), column sums over the device-side valid rows"""
    from nnr_b200 import ops
    g = torch.Generator().manual_seed(cols)
    cap, valid = 5000, 4321
    x = torch.randn(cap, cols, generator=g).to(cuda)
    r_dev = torch.tensor([valid], dtype=torch.int32, device=cuda)
    ref_pl = ops.tc_split(x, cap, cols, cols, r_dev)
    out = torch.full((cols,), float('nan'), device=cuda)
    pl = ops.tc_split(x, cap, cols, cols, r_dev, colsum_out=out)
    rows_w = (valid + 63) // 64 * 64
    pitch = pl.pitch
    a = ref_pl.buf.view(torch.int16).view(2, cap, pitch)[:, :rows_w]
    b = pl.buf.view(torch.int16).view(2, cap, pitch)[:, :rows_w]
    assert torch.equal(a, b)
    ref = x[:valid].double().sum(0)
    assert (out.double() - ref).abs().max().item() < 1e-3 * ref.abs().max().item() + 1e-3
    out2 = out.clone()
    ops.tc_split(x, cap, cols, cols, r_dev, colsum_out=out2, accumulate=True)
    assert torch.allclose(out2, 2 * out, rtol=1e-6, atol=1e-6)
    out3 = torch.empty_like(out)
    ops.tc_split(x, cap, cols, cols, r_dev, colsum_out=out3)
    assert torch.equal(out3, out)                                  # deterministic


@pytest.mark.parametrize('M,m_valid', [(1000, 1000), (1000, 333), (40000, 38017)])     # the last one runs on CTA pairs
def test_result_also_written_as_operand_planes(cuda, M, m_valid):
    """nnr_gemm_args.C_planes: the epilogue writes the result a second time as bf16 hi / lo operand planes -- bit for bit what
    nnr_tc_split of the fp32 result produces, rows [m, round_up(m, 64)) zeroed -- for the gate epilogue and the plain one"""
    from nnr_b200 import ops
    if ops.default_algo() not in (ops.ALGO_BF16, ops.ALGO_BF16X3):
        pytest.skip('operand planes of the bf16 tensor-core algorithms')
    g = torch.Generator().manual_seed(M + m_valid)
    N, K, R = 400, 400, 57
    A = torch.randn(M, K, generator=g).to(cuda)
    W = (torch.randn(N, K, generator=g) / 20).to(cuda)
    m_dev = torch.tensor([m_valid], dtype=torch.int32, device=cuda)
    rowbias = torch.randn(R, N, generator=g).to(cuda)
    rowmap = torch.randint(0, R, (M,), generator=g, dtype=torch.int32).to(cuda)
    aux = torch.randn(M, N, generator=g).to(cuda)
    for epi, kw in ((ops.EPI_NONE, {}),
                    (ops.EPI_GATE, dict(rowbias=rowbias, ldrowbias=N, rowmap=rowmap, aux=aux, ldaux=N,
                                        aux_out=torch.empty(M, N, device=cuda), ldaux_out=N))):
        C0 = torch.zeros(M, N, device=cuda)
        ops.gemm(A, W, C0, M, N, K, K, K, N, False, True, epi, m_dev=m_dev, **kw)
        C1 = torch.zeros(M, N, device=cuda)
        pl = ops.planes_empty(M, N, cuda)
        pl.buf.fill_(0x7f)
        ops.gemm(A, W, C1, M, N, K, K, K, N, False, True, epi, m_dev=m_dev, c_planes=pl, **kw)
        assert torch.equal(C0, C1)
        ref = ops.tc_split(C1, M, N, N, m_dev)
        rows = min(M, (m_valid + 63) // 64 * 64)
        npl = ref.buf.numel() // (M * ref.pitch * ref.esz)
        assert torch.equal(ref.buf.view(npl, M, -1)[:, :rows], pl.buf.view(npl, M, -1)[:, :rows]), (M, m_valid, epi)
