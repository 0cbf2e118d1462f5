"""torch-level wrappers over the C-ABI (``_lib``), registered as ``torch.ops.nnr.*`` custom ops.

Every op is an out-variant: the caller (PyTorch's caching allocator) owns all buffers, the library
only launches kernels on the current CUDA stream.  Ops are registered for the CUDA dispatch key
only -- calling them with CPU tensors raises (there is no CPU fallback by design).
"""
import ctypes as C

import torch

from . import _lib
from ._lib import GemmArgs, PoolArgs, check, lib

EPI_NONE, EPI_BIAS, EPI_BIAS_TANH, EPI_BIAS_RELU_RES, EPI_GATE, EPI_ADD_AUX = range(6)
ALGO_AUTO, ALGO_SIMT, ALGO_TF32X3, ALGO_BF16, ALGO_BF16X3 = range(5)

_F32, _I32, _I64, _U8 = torch.float32, torch.int32, torch.int64, torch.uint8


def _p(t, dtype=None):
    """device pointer of a tensor (None -> NULL) with device/dtype checks"""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError('nnr_b200 ops need CUDA tensors (no CPU fallback)')
    if dtype is not None and t.dtype != dtype:
        if not (dtype == _U8 and t.dtype == torch.bool):
            raise RuntimeError('nnr_b200: expected %s, got %s' % (dtype, t.dtype))
    return t.data_ptr()


_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None)


def _stream():
    """cudaStream_t of torch's current stream (raw handle: torch.cuda.current_stream() costs ~10 us per call, and a
    training step makes a few hundred launches)"""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


_ws_cache = {}
lane = 0      # engine.Lanes: index of the stream the caller is launching on (0 = the caller's own stream, 1 = the side lane)


def workspace(nbytes, device, tag='default'):
    """grow-only scratch buffer per (device, lane, tag); safe because all launches of one lane are stream ordered and
    concurrent lanes (engine.Lanes) never share a scratch buffer"""
    key = (device.index if device.index is not None else torch.cuda.current_device(), lane, tag)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


# --------------------------------------------------------------------------------------------
# implementations (plain python functions over tensors)
# --------------------------------------------------------------------------------------------
def seq_prepare(mask, len_, off, tok_row):
    N, L = mask.shape
    check(lib.nnr_seq_prepare(_p(mask, _U8), N, L, _p(len_, _I32), _p(off, _I32), _p(tok_row, _I32), _stream()),
          'nnr_seq_prepare')


def embed_gather_fwd(table, ids, len_, off, out, p_drop, seed):
    N, L = ids.shape
    V, E = table.shape
    check(lib.nnr_embed_gather_fwd(_p(table, _F32), _p(ids, _I32), _p(len_, _I32), _p(off, _I32), N, L, E, V,
                                   _p(out, _F32), float(p_drop), int(seed), _stream()), 'nnr_embed_gather_fwd')


def embed_gather_planes_fwd(table, ids, len_, off, cap, p_drop, seed):
    """embedding gather + dropout emitted as GEMM operand planes (no fp32 [tokens, E] tensor); tensor-core algos only"""
    N, L = ids.shape
    V, E = table.shape
    algo = default_algo()
    nbytes = int(lib.nnr_tc_split_bytes(cap, E, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=table.device)
    check(lib.nnr_embed_gather_planes_fwd(_p(table, _F32), _p(ids, _I32), _p(len_, _I32), _p(off, _I32), N, L, E, V, cap,
                                          float(p_drop), int(seed), algo, buf.data_ptr(), nbytes, _stream()),
          'nnr_embed_gather_planes_fwd')
    return Planes(buf, cap, E, int(lib.nnr_tc_split_pitch(E, algo)), 2 if algo in (ALGO_BF16, ALGO_BF16X3) else 4)


def embed_gather_bwd(dout, ids, len_, off, dtable, p_drop, seed, accumulate):
    N, L = ids.shape
    V, E = dtable.shape
    nbytes = lib.nnr_embed_gather_bwd_workspace_bytes(N, L)
    ws = workspace(nbytes, dout.device, 'embed')
    check(lib.nnr_embed_gather_bwd(_p(dout, _F32), _p(ids, _I32), _p(len_, _I32), _p(off, _I32), N, L, E, V,
                                   float(p_drop), int(seed), _p(dtable, _F32), int(accumulate), ws.data_ptr(),
                                   ws.numel(), _stream()), 'nnr_embed_gather_bwd')


class Planes:
    """Operand planes of the tensor-core GEMM backend (nnr_tc_split): fp32 [hi|lo][rows][pitch] for 3xTF32,
    bf16 [1][rows][pitch] for the bf16 variant.  ``cols(a, b)`` is a column-slice view (same planes)."""
    __slots__ = ('buf', 'rows', 'ncols', 'pitch', 'esz', 'col_off')

    def __init__(self, buf, rows, ncols, pitch, esz, col_off=0):
        self.buf, self.rows, self.ncols, self.pitch, self.esz, self.col_off = buf, rows, ncols, pitch, esz, col_off

    def ptr(self):
        return self.buf.data_ptr() + self.col_off * self.esz

    def cols(self, a, b):
        return Planes(self.buf, self.rows, b - a, self.pitch, self.esz, self.col_off + a)


def default_algo():
    return int(lib.nnr_gemm_default_algo())


def planes_empty(rows, cols, device):
    """uninitialised operand planes for a producer kernel to fill (bf16 tensor-core algos), or None"""
    algo = default_algo()
    if algo not in (ALGO_BF16, ALGO_BF16X3):
        return None
    buf = torch.empty(int(lib.nnr_tc_split_bytes(rows, cols, algo)), dtype=torch.uint8, device=device)
    return Planes(buf, rows, cols, int(lib.nnr_tc_split_pitch(cols, algo)), 2)


def tc_split(x, rows, cols, ld, r_dev=None, colsum_out=None, accumulate=False):
    """pre-split a row-major [rows, cols] fp32 matrix once so several GEMMs can share the planes; returns None
    when the exact-fp32 backend is selected (NNR_GEMM_ALGO=simt).  With ``colsum_out`` the column sums of the valid
    rows are produced by the same pass (nnr_tc_split_colsum)."""
    algo = default_algo()
    if algo == ALGO_SIMT:
        if colsum_out is not None:
            colsum(x, ld, rows, cols, colsum_out, accumulate, r_dev)
        return None
    nbytes = int(lib.nnr_tc_split_bytes(rows, cols, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    if colsum_out is not None and cols <= 2048 and ld % 4 == 0 and x.data_ptr() % 16 == 0:
        wsb = int(lib.nnr_tc_split_colsum_workspace_bytes(rows, cols, algo))
        ws = workspace(wsb, x.device, 'split_colsum')
        check(lib.nnr_tc_split_colsum(_p(x, _F32), ld, rows, cols, _p(r_dev, _I32), algo, buf.data_ptr(), nbytes,
                                      _p(colsum_out, _F32), int(accumulate), ws.data_ptr(), ws.numel(), _stream()),
              'nnr_tc_split_colsum')
        return Planes(buf, rows, cols, int(lib.nnr_tc_split_pitch(cols, algo)), 2 if algo in (ALGO_BF16, ALGO_BF16X3) else 4)
    if colsum_out is not None:
        colsum(x, ld, rows, cols, colsum_out, accumulate, r_dev)
    check(lib.nnr_tc_split(_p(x, _F32), ld, rows, cols, _p(r_dev, _I32), algo, buf.data_ptr(), nbytes, _stream()),
          'nnr_tc_split')
    return Planes(buf, rows, cols, int(lib.nnr_tc_split_pitch(cols, algo)), 2 if algo in (ALGO_BF16, ALGO_BF16X3) else 4)


def relu_bwd_split_colsum(dy, relu_out, rows, cols, p_drop, seed, dy_dropped, colsum_out):
    """planes of dy * dropout_mask * (relu_out > 0) + their column sums in one pass; dy_dropped (optional, not aliasing dy)
    receives dy * dropout_mask.  Tensor-core algos only."""
    algo = default_algo()
    nbytes = int(lib.nnr_tc_split_bytes(rows, cols, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=dy.device)
    wsb = int(lib.nnr_tc_split_colsum_workspace_bytes(rows, cols, algo))
    ws = workspace(wsb, dy.device, 'split_colsum')
    check(lib.nnr_relu_bwd_split_colsum(_p(dy, _F32), _p(relu_out, _F32), dy.stride(0), rows, cols, float(p_drop), int(seed),
                                        _p(dy_dropped, _F32), algo, buf.data_ptr(), nbytes, _p(colsum_out, _F32), 0,
                                        ws.data_ptr(), ws.numel(), _stream()), 'nnr_relu_bwd_split_colsum')
    return Planes(buf, rows, cols, int(lib.nnr_tc_split_pitch(cols, algo)), 2 if algo in (ALGO_BF16, ALGO_BF16X3) else 4)


class SplitMany:
    """operand planes of a fixed set of row-major matrices (the weight matrices), refreshed by ONE kernel launch"""

    def __init__(self, mats):
        import ctypes as C_
        from ._lib import SplitDesc
        self.algo = default_algo()
        self.planes = []
        self.n = 0
        if self.algo == ALGO_SIMT or not mats:
            return
        dev = mats[0].device
        arr = (SplitDesc * len(mats))()
        esz = 2 if self.algo in (ALGO_BF16, ALGO_BF16X3) else 4
        for i, w in enumerate(mats):
            rows, cols = w.shape
            pitch = int(lib.nnr_tc_split_pitch(cols, self.algo))
            buf = torch.empty(int(lib.nnr_tc_split_bytes(rows, cols, self.algo)), dtype=torch.uint8, device=dev)
            arr[i].src, arr[i].ld, arr[i].rows, arr[i].cols = w.data_ptr(), w.stride(0), rows, cols
            arr[i].planes, arr[i].pitch = buf.data_ptr(), pitch
            self.planes.append(Planes(buf, rows, cols, pitch, esz))
        raw = bytes(arr)
        self.descs = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
        self.n = len(mats)

    def refresh(self):
        if self.n:
            check(lib.nnr_tc_split_many(self.descs.data_ptr(), self.n, self.algo, _stream()), 'nnr_tc_split_many')


def gemm(A, B, Cout, M, N, K, lda, ldb, ldc, transA, transB, epilogue=EPI_NONE, accumulate=False, bias=None,
         aux=None, ldaux=0, aux_out=None, ldaux_out=0, rowbias=None, ldrowbias=0, rowmap=None, m_dev=None,
         k_dev=None, p_drop=0.0, seed=0, algo=ALGO_AUTO, a_planes=None, b_planes=None, c_planes=None):
    a = GemmArgs()
    a.A, a.lda, a.transA = _p(A, _F32), lda, int(transA)
    a.B, a.ldb, a.transB = _p(B, _F32), ldb, int(transB)
    a.C, a.ldc = _p(Cout, _F32), ldc
    a.M, a.N, a.K = M, N, K
    a.m_dev, a.k_dev = _p(m_dev, _I32), _p(k_dev, _I32)
    a.epilogue, a.accumulate = epilogue, int(accumulate)
    a.bias = _p(bias, _F32)
    a.aux, a.ldaux = _p(aux, _F32), ldaux
    a.aux_out, a.ldaux_out = _p(aux_out, _F32), ldaux_out
    a.rowbias, a.ldrowbias, a.rowmap = _p(rowbias, _F32), ldrowbias, _p(rowmap, _I32)
    a.p_drop, a.seed, a.algo = float(p_drop), int(seed), algo
    if a_planes is not None and algo == ALGO_AUTO:
        a.A_planes, a.a_planes_pitch, a.a_planes_rows = a_planes.ptr(), a_planes.pitch, a_planes.rows
    if b_planes is not None and algo == ALGO_AUTO:
        a.B_planes, a.b_planes_pitch, a.b_planes_rows = b_planes.ptr(), b_planes.pitch, b_planes.rows
    if c_planes is not None:
        a.C_planes, a.c_planes_pitch, a.c_planes_rows = c_planes.ptr(), c_planes.pitch, c_planes.rows
    nbytes = lib.nnr_gemm_workspace_bytes(C.byref(a))
    if nbytes:
        ws = workspace(nbytes, Cout.device, 'gemm')
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    check(lib.nnr_gemm(C.byref(a), _stream()), 'nnr_gemm')


def colsum(X, ldx, M, N, out, accumulate=False, m_dev=None):
    nbytes = lib.nnr_colsum_workspace_bytes(M, N)
    ws = workspace(nbytes, X.device, 'colsum')
    check(lib.nnr_colsum(_p(X, _F32), ldx, M, N, _p(m_dev, _I32), _p(out, _F32), int(accumulate), ws.data_ptr(),
                         ws.numel(), _stream()), 'nnr_colsum')


def length_sort_desc(len64, max_key):
    """sorted_idx of torch.sort(len64, descending=True) for small integer keys (stable: ties by original index)"""
    N = len64.numel()
    out = torch.empty(N, dtype=torch.int64, device=len64.device)
    check(lib.nnr_length_sort_desc(_p(len64, _I64), N, int(max_key), _p(out, _I64), _stream()), 'nnr_length_sort_desc')
    return out


def segment_colsum(X, ldx, off, N, D, out, ldo):
    check(lib.nnr_segment_colsum(_p(X, _F32), ldx, _p(off, _I32), N, D, _p(out, _F32), ldo, _stream()),
          'nnr_segment_colsum')


def _tile_counters(dev):
    return workspace(64, dev, 'lstm_counters').view(torch.int32)


def lstm_fwd(gx, w_hh, len_, off, order, N, L, H, h_out, c_stash, c_n):
    check(lib.nnr_lstm_fwd(_p(gx, _F32), _p(w_hh, _F32), _p(len_, _I32), _p(off, _I32), _p(order, _I32), N, L, H,
                           _p(h_out, _F32), _p(c_stash, _F32), _p(c_n, _F32), _tile_counters(gx.device).data_ptr(),
                           _stream()), 'nnr_lstm_fwd')


def lstm_fwd_planes_supported(H):
    return bool(lib.nnr_lstm_fwd_planes_supported(H, default_algo()))


def lstm_fwd_planes(gx, w_hh, len_, off, order, N, L, H, h_out, c_stash, c_n, cap):
    """lstm_fwd whose h also leaves as GEMM operand planes (returned): no split pass over h"""
    algo = default_algo()
    nbytes = int(lib.nnr_tc_split_bytes(cap, 2 * H, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=gx.device)
    check(lib.nnr_lstm_fwd_planes(_p(gx, _F32), _p(w_hh, _F32), _p(len_, _I32), _p(off, _I32), _p(order, _I32), N, L, H,
                                  _p(h_out, _F32), _p(c_stash, _F32), _p(c_n, _F32), _tile_counters(gx.device).data_ptr(), cap, algo,
                                  buf.data_ptr(), nbytes, _stream()), 'nnr_lstm_fwd_planes')
    return Planes(buf, cap, 2 * H, int(lib.nnr_tc_split_pitch(2 * H, algo)), 2)


def lstm_bwd(gates, c_stash, w_hh, len_, off, order, N, L, H, dh, dcn):
    check(lib.nnr_lstm_bwd(_p(gates, _F32), _p(c_stash, _F32), _p(w_hh, _F32), _p(len_, _I32), _p(off, _I32),
                           _p(order, _I32), N, L, H, _p(dh, _F32), _p(dcn, _F32), _tile_counters(gates.device).data_ptr(),
                           _stream()), 'nnr_lstm_bwd')


def lstm_bwd_planes_supported(H):
    return bool(lib.nnr_lstm_bwd_planes_supported(H, default_algo()))


def lstm_bwd_planes(gates, c_stash, w_hh, len_, off, order, N, L, H, dh, dcn, cap, db):
    """BPTT whose dL/dgx leaves as GEMM operand planes (returned) and whose column sums land in db [8H]"""
    algo = default_algo()
    nbytes = int(lib.nnr_tc_split_bytes(cap, 8 * H, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=gates.device)
    wsb = int(lib.nnr_lstm_bwd_planes_workspace_bytes(N, H))
    ws = workspace(wsb, gates.device, 'lstm_db')
    check(lib.nnr_lstm_bwd_planes(_p(gates, _F32), _p(c_stash, _F32), _p(w_hh, _F32), _p(len_, _I32), _p(off, _I32),
                                  _p(order, _I32), N, L, H, _p(dh, _F32), _p(dcn, _F32),
                                  _tile_counters(gates.device).data_ptr(), cap, algo, buf.data_ptr(), nbytes, _p(db, _F32),
                                  ws.data_ptr(), ws.numel(), _stream()), 'nnr_lstm_bwd_planes')
    return Planes(buf, cap, 8 * H, int(lib.nnr_tc_split_pitch(8 * H, algo)), 2)


def lstm_shift_h(h, len_, off, tok_row, N, L, H, hprev):
    check(lib.nnr_lstm_shift_h(_p(h, _F32), _p(len_, _I32), _p(off, _I32), _p(tok_row, _I32), N, L, H,
                               _p(hprev, _F32), _stream()), 'nnr_lstm_shift_h')


def lstm_shift_h_planes(h, len_, off, tok_row, N, L, H, cap):
    """hprev (nnr_lstm_shift_h) emitted as GEMM operand planes; tensor-core algos only"""
    algo = default_algo()
    nbytes = int(lib.nnr_tc_split_bytes(cap, 2 * H, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=h.device)
    check(lib.nnr_lstm_shift_h_planes(_p(h, _F32), _p(len_, _I32), _p(off, _I32), _p(tok_row, _I32), N, L, H, cap, algo,
                                      buf.data_ptr(), nbytes, _stream()), 'nnr_lstm_shift_h_planes')
    return Planes(buf, cap, 2 * H, int(lib.nnr_tc_split_pitch(2 * H, algo)), 2 if algo in (ALGO_BF16, ALGO_BF16X3) else 4)


def gate_bwd_pre(dhg, h, g, n_max, n_dev, D, dz, dh0):
    check(lib.nnr_gate_bwd_pre(_p(dhg, _F32), _p(h, _F32), _p(g, _F32), n_max, _p(n_dev, _I32), D, _p(dz, _F32),
                               _p(dh0, _F32), _stream()), 'nnr_gate_bwd_pre')


def gate_bwd_planes(dhg, h, g, off, N, D, cap, dh0, dmproj):
    """selective-gate backward prologue with dz emitted as GEMM operand planes and its per-news sums in dmproj"""
    algo = default_algo()
    nbytes = int(lib.nnr_tc_split_bytes(cap, D, algo))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=h.device)
    check(lib.nnr_gate_bwd_planes(_p(dhg, _F32), _p(h, _F32), _p(g, _F32), _p(off, _I32), N, D, cap, algo, buf.data_ptr(),
                                  nbytes, _p(dh0, _F32), _p(dmproj, _F32), dmproj.stride(0), _stream()), 'nnr_gate_bwd_planes')
    return Planes(buf, cap, D, int(lib.nnr_tc_split_pitch(D, algo)), 2 if algo in (ALGO_BF16, ALGO_BF16X3) else 4)


def _pool_args(X, ldx, D, S, max_len, mode, seg_off=None, fixed_len=0, U=None, ldu=0, A=0, w2=None, qvec=None,
               ldq=0, scale=1.0, mask=None, pooled=None, ldp=0, alpha=None, dpooled=None, lddp=0, dX=None, lddx=0,
               accumulate_dx=False, dU=None, lddu=0, dw2_partial=None, dqvec=None, lddq=0, seg_order=None):
    a = PoolArgs()
    a.X, a.ldx, a.D = _p(X, _F32), ldx, D
    a.seg_off, a.S, a.fixed_len, a.max_len = _p(seg_off, _I32), S, fixed_len, max_len
    a.mode = mode
    a.U, a.ldu, a.A, a.w2 = _p(U, _F32), ldu, A, _p(w2, _F32)
    a.qvec, a.ldq, a.scale = _p(qvec, _F32), ldq, float(scale)
    a.mask = _p(mask, _U8)
    a.pooled, a.ldp = _p(pooled, _F32), ldp
    a.alpha = _p(alpha, _F32)
    a.dpooled, a.lddp = _p(dpooled, _F32), lddp
    a.dX, a.lddx, a.accumulate_dx = _p(dX, _F32), lddx, int(accumulate_dx)
    a.seg_order = _p(seg_order, _I32)
    a.dU, a.lddu = _p(dU, _F32), lddu
    a.dw2_partial = _p(dw2_partial, _F32)
    a.dqvec, a.lddq = _p(dqvec, _F32), lddq
    return a


def attn_pool_fwd(**kw):
    a = _pool_args(**kw)
    check(lib.nnr_attn_pool_fwd(C.byref(a), _stream()), 'nnr_attn_pool_fwd')


def attn_pool_bwd(**kw):
    a = _pool_args(**kw)
    check(lib.nnr_attn_pool_bwd(C.byref(a), _stream()), 'nnr_attn_pool_bwd')


def news_fuse_fwd(ts, tc, cs, cc, cat_table, sub_table, cat, sub, N, D2, p_drop, seed, out):
    Ec, Es = cat_table.shape[1], sub_table.shape[1]
    check(lib.nnr_news_fuse_fwd(_p(ts, _F32), _p(tc, _F32), _p(cs, _F32), _p(cc, _F32), _p(cat_table, _F32),
                                _p(sub_table, _F32), _p(cat, _I32), _p(sub, _I32), N, D2, Ec, Es, float(p_drop),
                                int(seed), _p(out, _F32), _stream()), 'nnr_news_fuse_fwd')


def news_fuse_bwd(dout, cat, sub, N, D2, p_drop, seed, d_a, d_b, dcat_table, dsub_table, accumulate):
    Ec, Es = dcat_table.shape[1], dsub_table.shape[1]
    check(lib.nnr_news_fuse_bwd(_p(dout, _F32), _p(cat, _I32), _p(sub, _I32), N, D2, Ec, Es, dcat_table.shape[0],
                                dsub_table.shape[0], float(p_drop), int(seed), _p(d_a, _F32), _p(d_b, _F32),
                                _p(dcat_table, _F32), _p(dsub_table, _F32), int(accumulate), _stream()),
          'nnr_news_fuse_bwd')


def news_fuse_split_bwd(dout, N, D2, Ec, Es, d_a, d_b):
    """the activation half of news_fuse_bwd: d_a = dout[:, :D2], d_b = dout[:, D2:2*D2]"""
    check(lib.nnr_news_fuse_bwd(_p(dout, _F32), None, None, N, D2, Ec, Es, 0, 0, 0.0, 0, _p(d_a, _F32), _p(d_b, _F32), None, None, 0,
                                _stream()), 'nnr_news_fuse_bwd')


def news_fuse_tables_bwd(dout, cat, sub, N, col0, p_drop, seed, dcat_table, dsub_table, accumulate):
    """the table-gradient half of news_fuse_bwd (a leaf of the backward pass: the engine issues it on a side lane)"""
    Ec, Es = dcat_table.shape[1], dsub_table.shape[1]
    check(lib.nnr_news_fuse_tables_bwd(_p(dout, _F32), _p(cat, _I32), _p(sub, _I32), N, dout.shape[1], col0, Ec, Es,
                                       dcat_table.shape[0], dsub_table.shape[0], float(p_drop), int(seed), _p(dcat_table, _F32),
                                       _p(dsub_table, _F32), int(accumulate), _stream()), 'nnr_news_fuse_tables_bwd')


GRAPH_NO_SELF_CONNECTION, GRAPH_NO_NORMALIZATION, GRAPH_ASYMMETRIC = 1, 2, 4


def graph_flags(no_self_connection=False, no_adjacent_normalization=False, gcn_normalization_type='symmetric'):
    """the reference's graph options (config.py:56-58) as the flag word of nnr_sue_graph_build_ex"""
    return ((GRAPH_NO_SELF_CONNECTION if no_self_connection else 0) | (GRAPH_NO_NORMALIZATION if no_adjacent_normalization else 0)
            | (GRAPH_ASYMMETRIC if gcn_normalization_type == 'asymmetric' else 0))


def sue_graph_build(categories, history_len, C_num, graph=None, category_mask=None, category_indices=None, flags=0):
    B, H = categories.shape
    check(lib.nnr_sue_graph_build_ex(_p(categories, _I32), _p(history_len, _I32), B, H, C_num, int(flags), _p(graph, _F32),
                                     _p(category_mask, _U8), _p(category_indices, _I64), _stream()), 'nnr_sue_graph_build')


def ln_relu_res_fwd(y, gamma, beta, res, R, D, eps, p_drop, seed, out, relu_out, mean, rstd):
    check(lib.nnr_ln_relu_res_fwd(_p(y, _F32), _p(gamma, _F32), _p(beta, _F32), _p(res, _F32), R, D, float(eps), float(p_drop),
                                  int(seed), _p(out, _F32), _p(relu_out, _F32), _p(mean, _F32), _p(rstd, _F32), _stream()),
          'nnr_ln_relu_res_fwd')


def ln_relu_res_bwd(dout, y, gamma, relu_out, mean, rstd, R, D, p_drop, seed, dout_dropped, dy, dgamma, dbeta):
    nbytes = lib.nnr_ln_relu_res_bwd_workspace_bytes(R, D)
    ws = workspace(nbytes, dout.device, 'ln')
    check(lib.nnr_ln_relu_res_bwd(_p(dout, _F32), _p(y, _F32), _p(gamma, _F32), _p(relu_out, _F32), _p(mean, _F32), _p(rstd, _F32),
                                  R, D, float(p_drop), int(seed), _p(dout_dropped, _F32), _p(dy, _F32), _p(dgamma, _F32),
                                  _p(dbeta, _F32), ws.data_ptr(), ws.numel(), _stream()), 'nnr_ln_relu_res_bwd')


def graph_to_csr(graph, transpose, nnz, col, val):
    B, G, _ = graph.shape
    check(lib.nnr_graph_to_csr(_p(graph, _F32), B, G, int(transpose), _p(nnz, _I32), _p(col, _I32), _p(val, _F32),
                               _stream()), 'nnr_graph_to_csr')


def gcn_aggregate(nnz, col, val, x, B, G, D, out, add=None):
    """out = A x (+ add: the residual term of the backward, same pass)"""
    if add is not None:
        check(lib.nnr_gcn_aggregate_add(_p(nnz, _I32), _p(col, _I32), _p(val, _F32), _p(x, _F32), B, G, D, _p(add, _F32),
                                        _p(out, _F32), _stream()), 'nnr_gcn_aggregate_add')
        return
    check(lib.nnr_gcn_aggregate(_p(nnz, _I32), _p(col, _I32), _p(val, _F32), _p(x, _F32), B, G, D, _p(out, _F32),
                                _stream()), 'nnr_gcn_aggregate')


def cluster_intra_fwd(Kp, Qp, g, idx, B, n, H, Au, D, C1, scale, alpha, intra):
    check(lib.nnr_cluster_intra_fwd(_p(Kp, _F32), _p(Qp, _F32), _p(g, _F32), _p(idx, _I64), B, n, H, Au, D, C1,
                                    float(scale), _p(alpha, _F32), _p(intra, _F32), _stream()), 'nnr_cluster_intra_fwd')


def cluster_intra_bwd(dintra, Kp, Qp, g, idx, alpha, B, n, H, Au, D, C1, scale, da_ws, dKp, dQp, dg, accumulate_dg):
    check(lib.nnr_cluster_intra_bwd(_p(dintra, _F32), _p(Kp, _F32), _p(Qp, _F32), _p(g, _F32), _p(idx, _I64),
                                    _p(alpha, _F32), B, n, H, Au, D, C1, float(scale), _p(da_ws, _F32), _p(dKp, _F32),
                                    _p(dQp, _F32), _p(dg, _F32), int(accumulate_dg), _stream()), 'nnr_cluster_intra_bwd')


def cluster_tail_scores(Kp, g, Wg, idx, cmask, Qp, qk2, cand, bias, B, H, Au, D, C1, T, scale, scores):
    """click scores [B, T] (row stride scores.stride(0)) of T candidates shared by B users through the factored cluster tail
    (nnr_cluster_tail_scores)"""
    check(lib.nnr_cluster_tail_scores(_p(Kp, _F32), _p(g, _F32), _p(Wg, _F32), _p(idx, _I64), _p(cmask, _U8), _p(Qp, _F32),
                                      _p(qk2, _F32), _p(cand, _F32), _p(bias, _F32), B, H, Au, D, C1, T, float(scale),
                                      _p(scores, _F32), scores.stride(0), _stream()), 'nnr_cluster_tail_scores')


def cluster_tail_scores_packed(Kp, g, Wg, idx, cmask, row_off, Qp, qk2, cand, bias, B, H, Au, D, C1, n_max, scale, scores):
    """click scores [B, n_max] (row stride scores.stride(0)) of per-user candidate lists: user b's are rows
    [row_off[b], row_off[b + 1]) of Qp / qk2 / cand (Qp.shape[0] rows), through the factored cluster tail; entries past a
    user's count are left as they are (nnr_cluster_tail_scores_packed)"""
    check(lib.nnr_cluster_tail_scores_packed(_p(Kp, _F32), _p(g, _F32), _p(Wg, _F32), _p(idx, _I64), _p(cmask, _U8),
                                             _p(row_off, _I32), Qp.shape[0], _p(Qp, _F32), _p(qk2, _F32), _p(cand, _F32),
                                             _p(bias, _F32), B, H, Au, D, C1, n_max, float(scale), _p(scores, _F32),
                                             scores.stride(0), _stream()), 'nnr_cluster_tail_scores_packed')


def rowdot_fwd(a, b, R, D, out):
    check(lib.nnr_rowdot_fwd(_p(a, _F32), _p(b, _F32), R, D, _p(out, _F32), _stream()), 'nnr_rowdot_fwd')


def rowdot_bwd(dout, a, b, R, D, da, accumulate_a, db, accumulate_b):
    check(lib.nnr_rowdot_bwd(_p(dout, _F32), _p(a, _F32), _p(b, _F32), R, D, _p(da, _F32), int(accumulate_a),
                             _p(db, _F32), int(accumulate_b), _stream()), 'nnr_rowdot_bwd')


TOPK_MAX_K, TOPK_MAX_TILE, TOPK_MAX_EXCLUDE, TOPK_MAX_GROUPS = 1024, 4096, 1024, 1024     # include/nnr_b200.h: NNR_TOPK_MAX_*


def topk_merge(scores, pos0, tile_ids, exclude, exclude_len, init, best_score, best_pos):
    """merge the score tile scores [B, T] (pool positions pos0 + j) into the running best list best_score / best_pos
    [B, k], skipping entries whose id tile_ids[j] is among the row's exclude[b, :exclude_len[b]] (nnr_topk_merge)"""
    B, T = scores.shape
    ldx = exclude.shape[1] if exclude is not None else 0
    check(lib.nnr_topk_merge(_p(scores, _F32), scores.stride(0), B, T, int(pos0), _p(tile_ids, _I64), _p(exclude, _I64),
                             _p(exclude_len, _I32), ldx, best_score.shape[1], int(init), _p(best_score, _F32),
                             _p(best_pos, _I64), _stream()), 'nnr_topk_merge')


def topk_merge_capped(scores, pos0, tile_ids, exclude, exclude_len, id_group, num_groups, cap, init, best_score, best_pos,
                      best_group):
    """topk_merge keeping at most ``cap`` entries per group: entry j's group is id_group[tile_ids[j]] (int32, in
    [0, num_groups)), best_group [B, k] int32 holds each list entry's group (nnr_topk_merge_capped)"""
    B, T = scores.shape
    ldx = exclude.shape[1] if exclude is not None else 0
    check(lib.nnr_topk_merge_capped(_p(scores, _F32), scores.stride(0), B, T, int(pos0), _p(tile_ids, _I64),
                                    _p(exclude, _I64), _p(exclude_len, _I32), ldx, best_score.shape[1], int(init),
                                    _p(id_group, _I32), int(num_groups), int(cap), _p(best_score, _F32), _p(best_pos, _I64),
                                    _p(best_group, _I32), _stream()), 'nnr_topk_merge_capped')


def topk_merge_lists(scores, pos, init, best_score, best_pos):
    """merge entries scores [B, T] whose pool positions are pos [B, T] (int64; < 0: an empty slot, skipped) into the running
    best list best_score / best_pos [B, k]: folds best lists of disjoint position sets into one (nnr_topk_merge_lists)"""
    B, T = scores.shape
    check(lib.nnr_topk_merge_lists(_p(scores, _F32), scores.stride(0), B, T, _p(pos, _I64), pos.stride(0),
                                   best_score.shape[1], int(init), _p(best_score, _F32), _p(best_pos, _I64), _stream()),
          'nnr_topk_merge_lists')


def topk_merge_lists_capped(scores, pos, grp, num_groups, cap, init, best_score, best_pos, best_group):
    """topk_merge_lists keeping at most ``cap`` entries per group: entry (b, j)'s group is grp[b, j] (int32, in
    [0, num_groups)), best_group [B, k] int32 holds each list entry's group (nnr_topk_merge_lists_capped)"""
    B, T = scores.shape
    check(lib.nnr_topk_merge_lists_capped(_p(scores, _F32), scores.stride(0), B, T, _p(pos, _I64), pos.stride(0),
                                          _p(grp, _I32), grp.stride(0), int(num_groups), int(cap), best_score.shape[1],
                                          int(init), _p(best_score, _F32), _p(best_pos, _I64), _p(best_group, _I32),
                                          _stream()), 'nnr_topk_merge_lists_capped')


def dropout(x, p_drop, seed, y):
    check(lib.nnr_dropout(_p(x, _F32), x.numel(), float(p_drop), int(seed), _p(y, _F32), _stream()), 'nnr_dropout')


def flat_clip_adam(param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, max_norm, grad_scale, step, norm_out):
    n = param.numel()
    nbytes = lib.nnr_flat_clip_adam_workspace_bytes(n)
    ws = workspace(nbytes, param.device, 'adam')
    check(lib.nnr_flat_clip_adam(_p(param, _F32), _p(grad, _F32), _p(exp_avg, _F32), _p(exp_avg_sq, _F32), n, lr,
                                 beta1, beta2, eps, max_norm, grad_scale, int(step), _p(norm_out, _F32),
                                 ws.data_ptr(), ws.numel(), _stream()), 'nnr_flat_clip_adam')


def flat_clip_adam_dev(param, grad, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, max_norm, grad_scale, step_dev, norm_out):
    """nnr_flat_clip_adam with the step counter on the device (int32 tensor, incremented by the call): graph-capturable"""
    n = param.numel()
    nbytes = lib.nnr_flat_clip_adam_workspace_bytes(n)
    ws = workspace(nbytes, param.device, 'adam')
    check(lib.nnr_flat_clip_adam_dev(_p(param, _F32), _p(grad, _F32), _p(exp_avg, _F32), _p(exp_avg_sq, _F32), n, lr,
                                     beta1, beta2, eps, max_norm, grad_scale, _p(step_dev, _I32), _p(norm_out, _F32),
                                     ws.data_ptr(), ws.numel(), _stream()), 'nnr_flat_clip_adam_dev')


# --------------------------------------------------------------------------------------------
# registration as torch custom ops (torch.ops.nnr.*), CUDA dispatch key only
# --------------------------------------------------------------------------------------------
_torch_lib = torch.library.Library('nnr', 'DEF')
_SCHEMAS = {
    'seq_prepare': ('(Tensor(a!) mask, Tensor(b!) len, Tensor(c!) off, Tensor(d!) tok_row) -> ()', seq_prepare),
    'embed_gather_fwd': ('(Tensor table, Tensor ids, Tensor len, Tensor off, Tensor(a!) out, float p_drop, int seed) -> ()',
                         embed_gather_fwd),
    'embed_gather_bwd': ('(Tensor dout, Tensor ids, Tensor len, Tensor off, Tensor(a!) dtable, float p_drop, int seed, '
                         'bool accumulate) -> ()', embed_gather_bwd),
    'lstm_fwd': ('(Tensor(a!) gx, Tensor w_hh, Tensor len, Tensor off, Tensor order, int N, int L, int H, '
                 'Tensor(b!) h_out, Tensor(c!) c_stash, Tensor(d!) c_n) -> ()', lstm_fwd),
    'lstm_bwd': ('(Tensor(a!) gates, Tensor c_stash, Tensor w_hh, Tensor len, Tensor off, Tensor order, int N, int L, '
                 'int H, Tensor dh, Tensor dcn) -> ()', lstm_bwd),
    'lstm_shift_h': ('(Tensor h, Tensor len, Tensor off, Tensor tok_row, int N, int L, int H, Tensor(a!) hprev) -> ()',
                     lstm_shift_h),
    'gcn_aggregate': ('(Tensor nnz, Tensor col, Tensor val, Tensor x, int B, int G, int D, Tensor(a!) out, Tensor? add=None) -> ()',
                      gcn_aggregate),
    'graph_to_csr': ('(Tensor graph, bool transpose, Tensor(a!) nnz, Tensor(b!) col, Tensor(c!) val) -> ()', graph_to_csr),
    'sue_graph_build': ('(Tensor categories, Tensor history_len, int C_num, Tensor(a!)? graph=None, Tensor(b!)? category_mask=None, '
                        'Tensor(c!)? category_indices=None, int flags=0) -> ()', sue_graph_build),
    'cluster_intra_fwd': ('(Tensor Kp, Tensor Qp, Tensor g, Tensor idx, int B, int n, int H, int Au, int D, int C1, '
                          'float scale, Tensor(a!) alpha, Tensor(b!) intra) -> ()', cluster_intra_fwd),
    'cluster_intra_bwd': ('(Tensor dintra, Tensor Kp, Tensor Qp, Tensor g, Tensor idx, Tensor alpha, int B, int n, int H, int Au, int D, '
                          'int C1, float scale, Tensor(a!) da_ws, Tensor(b!) dKp, Tensor(c!) dQp, Tensor(d!) dg, bool accumulate_dg) -> ()',
                          cluster_intra_bwd),
    'cluster_tail_scores': ('(Tensor Kp, Tensor g, Tensor Wg, Tensor idx, Tensor cmask, Tensor Qp, Tensor qk2, Tensor cand, '
                            'Tensor bias, int B, int H, int Au, int D, int C1, int T, float scale, Tensor(a!) scores) -> ()',
                            cluster_tail_scores),
    'cluster_tail_scores_packed': ('(Tensor Kp, Tensor g, Tensor Wg, Tensor idx, Tensor cmask, Tensor row_off, Tensor Qp, '
                                   'Tensor qk2, Tensor cand, Tensor bias, int B, int H, int Au, int D, int C1, int n_max, '
                                   'float scale, Tensor(a!) scores) -> ()', cluster_tail_scores_packed),
    'rowdot_fwd': ('(Tensor a, Tensor b, int R, int D, Tensor(a!) out) -> ()', rowdot_fwd),
    'rowdot_bwd': ('(Tensor dout, Tensor a, Tensor b, int R, int D, Tensor(a!) da, bool accumulate_a, Tensor(b!) db, bool accumulate_b) -> ()',
                   rowdot_bwd),
    'news_fuse_fwd': ('(Tensor ts, Tensor? tc, Tensor? cs, Tensor? cc, Tensor cat_table, Tensor sub_table, Tensor cat, Tensor sub, int N, '
                      'int D2, float p_drop, int seed, Tensor(a!) out) -> ()', news_fuse_fwd),
    'news_fuse_bwd': ('(Tensor dout, Tensor cat, Tensor sub, int N, int D2, float p_drop, int seed, Tensor(a!) d_a, Tensor(b!)? d_b, '
                      'Tensor(c!) dcat_table, Tensor(d!) dsub_table, bool accumulate) -> ()', news_fuse_bwd),
    'news_fuse_split_bwd': ('(Tensor dout, int N, int D2, int Ec, int Es, Tensor(a!) d_a, Tensor(b!)? d_b) -> ()', news_fuse_split_bwd),
    'news_fuse_tables_bwd': ('(Tensor dout, Tensor cat, Tensor sub, int N, int col0, float p_drop, int seed, Tensor(a!) dcat_table, '
                             'Tensor(b!) dsub_table, bool accumulate) -> ()', news_fuse_tables_bwd),
    'colsum': ('(Tensor X, int ldx, int M, int N, Tensor(a!) out, bool accumulate=False, Tensor? m_dev=None) -> ()', colsum),
    'segment_colsum': ('(Tensor X, int ldx, Tensor off, int N, int D, Tensor(a!) out, int ldo) -> ()', segment_colsum),
    'gate_bwd_pre': ('(Tensor dhg, Tensor h, Tensor g, int n_max, Tensor n_dev, int D, Tensor(a!) dz, Tensor(b!) dh0) -> ()', gate_bwd_pre),
    'ln_relu_res_fwd': ('(Tensor y, Tensor gamma, Tensor beta, Tensor? res, int R, int D, float eps, float p_drop, int seed, Tensor(a!) out, '
                        'Tensor(b!) relu_out, Tensor(c!) mean, Tensor(d!) rstd) -> ()', ln_relu_res_fwd),
    'ln_relu_res_bwd': ('(Tensor dout, Tensor y, Tensor gamma, Tensor relu_out, Tensor mean, Tensor rstd, int R, int D, float p_drop, int seed, '
                        'Tensor(a!)? dout_dropped, Tensor(b!) dy, Tensor(c!) dgamma, Tensor(d!) dbeta) -> ()', ln_relu_res_bwd),
    'dropout': ('(Tensor x, float p_drop, int seed, Tensor(a!) y) -> ()', dropout),
    'topk_merge': ('(Tensor scores, int pos0, Tensor? tile_ids, Tensor? exclude, Tensor? exclude_len, bool init, '
                   'Tensor(a!) best_score, Tensor(b!) best_pos) -> ()', topk_merge),
    'topk_merge_capped': ('(Tensor scores, int pos0, Tensor tile_ids, Tensor? exclude, Tensor? exclude_len, Tensor id_group, '
                          'int num_groups, int cap, bool init, Tensor(a!) best_score, Tensor(b!) best_pos, '
                          'Tensor(c!) best_group) -> ()', topk_merge_capped),
    'topk_merge_lists': ('(Tensor scores, Tensor pos, bool init, Tensor(a!) best_score, Tensor(b!) best_pos) -> ()',
                         topk_merge_lists),
    'topk_merge_lists_capped': ('(Tensor scores, Tensor pos, Tensor grp, int num_groups, int cap, bool init, '
                                'Tensor(a!) best_score, Tensor(b!) best_pos, Tensor(c!) best_group) -> ()',
                                topk_merge_lists_capped),
    'flat_clip_adam': ('(Tensor(a!) param, Tensor grad, Tensor(b!) exp_avg, Tensor(c!) exp_avg_sq, float lr, float beta1, '
                       'float beta2, float eps, float max_norm, float grad_scale, int step, Tensor(d!) norm_out) -> ()',
                       flat_clip_adam),
    'flat_clip_adam_dev': ('(Tensor(a!) param, Tensor grad, Tensor(b!) exp_avg, Tensor(c!) exp_avg_sq, float lr, float beta1, '
                           'float beta2, float eps, float max_norm, float grad_scale, Tensor(e!) step_dev, Tensor(d!) norm_out) -> ()',
                           flat_clip_adam_dev),
}


def _noop(*a, **k):
    return None


for _name, (_schema, _fn) in _SCHEMAS.items():
    _torch_lib.define(_name + _schema)
    _torch_lib.impl(_name, _fn, 'CUDA')
    _torch_lib.impl(_name, _noop, 'Meta')


def _via_dispatcher(name):
    op = getattr(torch.ops.nnr, name)

    def call(*a, **k):
        return op(*a, **k)
    call.__name__ = name
    call.__doc__ = 'torch.ops.nnr.%s (CUDA dispatch key) -> %s' % (name, _SCHEMAS[name][1].__doc__ or 'C-ABI nnr_' + name)
    return call


# The engine reaches these ops through PyTorch's dispatcher (torch.ops.nnr.*): module attributes are rebound to dispatcher
# calls, the registered CUDA implementations are the ctypes wrappers above.
# Ops whose arguments are argument STRUCTS of the C ABI (nnr_gemm, nnr_attn_pool_*) or that return operand-plane handles
# (tc_split*, *_planes*) are plain functions: a dispatcher schema cannot carry them.
DISPATCHED = sorted(_SCHEMAS)
for _name in DISPATCHED:
    globals()[_name] = _via_dispatcher(_name)

launch_count = _lib.launch_count
