"""Forward / backward schedules of the CNE news encoder and the SUE user encoder over the C-ABI ops.

Each encoder call is ONE ``torch.autograd.Function`` whose forward and backward are explicit
sequences of ``nnr_*`` kernel launches (no autograd graph inside, no ATen math on the per-token
tensors).  Host PyTorch is used only for allocation, the [N]-sized permutation bookkeeping
(``torch.sort`` exactly as the reference calls it, so tie-breaking matches on the same device) and
slicing of the small per-news tensors.

Reference spans: CNE = newsEncoders.py:102-141, SUE = userEncoders.py:68-98, GCN = layers.py:285-323.
"""
import math
import os
import weakref

import torch

from . import ops
from .ops import (EPI_ADD_AUX, EPI_BIAS, EPI_BIAS_RELU_RES, EPI_BIAS_TANH, EPI_GATE, EPI_NONE)

# torch.sort exactly as newsEncoders.py:112-115 calls it; tests swap in a stable sort on both sides
sort_fn = torch.sort

class SeedSource:
    """Device-resident base of the dropout seeds (include/nnr_b200.h: NNR_SEED_INDIRECT).  Inside a step every dropout
    site gets ``INDIRECT | site << 48 | address(base)``; ``advance()`` moves the base on the device (one tiny kernel on the
    current stream), so a CUDA graph that captured the step draws fresh masks on every replay while the backward of a step
    still sees the seeds of its forward."""
    INDIRECT = 1 << 62
    _GOLDEN = 0x9E3779B97F4A7C15 - (1 << 64)            # as a signed 64-bit increment

    def __init__(self, device):
        self.base = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).to(device)
        self.site = 0

    def advance(self):
        self.base.add_(self._GOLDEN)
        self.site = 0

    def next(self):
        self.site += 1
        assert self.site < (1 << 14)
        return self.INDIRECT | (self.site << 48) | self.base.data_ptr()


seed_source = None        # trainer.TrainStep installs a SeedSource while it runs / captures a graph-mode step


def fresh_seed():
    """seed for the counter-based dropout RNG: drawn from torch's CPU RNG stream (a 62-bit value), or an indirect
    device-side seed when a SeedSource is active"""
    if seed_source is not None:
        return seed_source.next()
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def _empty(shape, dev, dtype=torch.float32):
    return torch.empty(shape, dtype=dtype, device=dev)


# ------------------------------------------------------------------------------------------------
# Two-lane schedules
# ------------------------------------------------------------------------------------------------
# The title and the content branch of the news encoder are independent between their exchange points (the partner's final
# cell state before the selective gate, the partner's self-attention vector before the cross attention, and the mirror
# images of both in the backward pass), and so are the weight-gradient GEMMs of the user encoder and its candidate-side
# projections.  Many kernels of the step cannot fill 148 SMs on their own: the LSTM recurrences end in a tail that is as
# long as the longest sequence, the per-news and user-encoder GEMMs are one or two dozen CTAs.  `Lanes.run` therefore
# issues one branch on a side stream and the other on the caller's stream and joins them before the next exchange point;
# inside a captured step the two lanes become parallel branches of the CUDA graph.  NNR_LANES=0 (or
# engine.concurrent = False, used by the per-op profiler) issues everything on the caller's stream in the same order.
_LANES = os.environ.get('NNR_LANES', '1') != '0'
concurrent = True
_side_streams = {}


class Lanes:
    """lane 0 = the caller's stream; lanes 1, 2 = side streams of the device (lane 2 takes leaves -- work nothing on the
    critical path waits for -- so that they do not queue in front of the title branch on lane 1)"""
    NSIDE = 2

    def __init__(self, dev):
        self.on = _LANES and concurrent and dev.type == 'cuda'
        self.keep = []                      # tensors of one lane that another lane reads: alive until the next join
        self.used = set()
        if self.on:
            idx = dev.index if dev.index is not None else torch.cuda.current_device()
            self.main = torch.cuda.current_stream(idx)
            self.sides = _side_streams.get(idx)
            if self.sides is None:
                self.sides = _side_streams[idx] = [torch.cuda.Stream(device=idx) for _ in range(self.NSIDE)]
            if any(s == self.main for s in self.sides):      # nested use from a side lane itself: stay serial
                self.on = False

    def fork(self, lane=1, after=0):
        """side lane `lane` may start after everything issued so far on lane `after` (0 = the caller's stream)"""
        if self.on:
            self.sides[lane - 1].wait_stream(self.main if after == 0 else self.sides[after - 1])
            self.used.add(lane)

    def on_side(self, fn, *a, lane=1, **k):
        """issue fn on a side lane (no implicit fork / join)"""
        if not self.on:
            return fn(*a, **k)
        prev, ops.lane = ops.lane, lane
        try:
            with torch.cuda.stream(self.sides[lane - 1]):
                return fn(*a, **k)
        finally:
            ops.lane = prev

    def leaf(self, fn, *a, **k):
        """issue fn on lane 2, ordered after everything issued so far on the CURRENT lane: for work nothing on the critical
        path waits for (weight gradients); its results are valid after the next full join()"""
        if not self.on:
            return fn(*a, **k)
        cur = ops.lane
        if cur == 2:
            return fn(*a, **k)
        self.fork(2, after=cur)
        return self.on_side(fn, *a, lane=2, **k)

    def join(self, *which):
        """the caller's stream waits for the given side lanes (default: every lane forked since its last join)"""
        if self.on:
            for lane in sorted(which or self.used):
                if lane in self.used:
                    self.main.wait_stream(self.sides[lane - 1])
                    self.used.discard(lane)
        if not self.used:
            self.keep.clear()

    def run(self, fn_side, fn_main):
        """fork; fn_side on lane 1, fn_main on the caller's stream; join lane 1.  Returns (side result, main result)."""
        self.fork()
        a = self.on_side(fn_side)
        b = fn_main()
        self.join(1)
        return a, b


# ------------------------------------------------------------------------------------------------
# GEMM helpers (row-major; weights are nn.Linear layout [out, in])
# ------------------------------------------------------------------------------------------------
# Operand planes of WEIGHT matrices are split once per parameter version and shared by the forward and the dgrad
# GEMMs of every call until the parameters change.  In-place updates through torch bump ``_version``; the fused
# clip+Adam kernel writes through raw pointers, so trainer.TrainStep calls ``weights_changed()`` after it.
_weight_planes = {}
_weight_epoch = 0


# trainer.TrainStep registers a callback here: grads_ready(stage) is called from inside the backward pass as soon as a
# group of parameter gradients is final in the flat gradient buffer ('sue': the user encoder's own parameters, 'cne': every
# news-encoder parameter except the word table, 'table': the word-embedding gradient), so that the data-parallel reduction
# of that group can start while the rest of the backward pass is still running (the reference's DDP does the same with
# its gradient buckets, trainer.py:219,296-300).
grads_ready = None


def _notify(stage):
    if grads_ready is not None:
        grads_ready(stage)


def _param_grads(P, names, G):
    """Gradients of the parameters for the tail of an autograd.Function.backward.  When every parameter's ``.grad`` is a
    preallocated buffer managed by trainer.TrainStep (flat gradient buffer, marked ``_nnr_flat_grad``), the gradients
    are added into those buffers with ONE multi-tensor add and ``None`` is returned to autograd, instead of ~70
    per-parameter AccumulateGrad add kernels per step."""
    if _flat_grads(P, names):
        live = [k for k in names if G.get(k) is not None]    # None: already accumulated in place (embedding table)
        torch._foreach_add_([P[k].grad for k in live], [G[k] for k in live])
        return (None,) * len(names)
    return tuple(G.get(k) for k in names)


def _shared_split(x, rows, cols, colsum_out=None, m_dev=None):
    """operand planes of a small activation that feeds two GEMMs (and, with ``colsum_out``, its column sums = a bias
    gradient); ``m_dev``: an int32 device scalar, rows from it on are not read"""
    return ops.tc_split(x, rows, cols, x.stride(0), m_dev, colsum_out=colsum_out)


def _fused_relu_bwd(dy, cols):
    """nnr_relu_bwd_split_colsum applies: tensor-core GEMM planes in use, contiguous 16-byte aligned rows, <= 2048 columns"""
    return (ops.default_algo() != ops.ALGO_SIMT and cols <= 2048 and cols % 4 == 0 and dy.is_contiguous()
            and dy.data_ptr() % 16 == 0)


def _flat_grads(P, names):
    """every parameter's .grad is a view of trainer.TrainStep's flat gradient buffer"""
    return all(getattr(P[k], '_nnr_flat_grad', False) and P[k].grad is not None for k in names)


def weights_changed():
    global _weight_epoch
    _weight_epoch += 1
    _weight_planes.clear()


def install_weight_planes(W, planes):
    """register externally refreshed planes of W (trainer.TrainStep re-splits all weights in one launch per step)"""
    _weight_planes[id(W)] = ((_weight_epoch, W._version, W.data_ptr(), W.shape[0], W.shape[1], W.stride(0)), planes, weakref.ref(W))


def weight_planes(W):
    # only nn.Parameter objects: a temporary (e.g. a torch.cat of two weights) can be freed and its address reused by a
    # different matrix of the same shape within one parameter version
    if not (isinstance(W, torch.nn.Parameter) or (W.is_leaf and W.requires_grad)) or W.dim() != 2 or W.stride(1) != 1 or not W.is_cuda:
        return None
    key = id(W)
    tag = (_weight_epoch, W._version, W.data_ptr(), W.shape[0], W.shape[1], W.stride(0))
    hit = _weight_planes.get(key)
    if hit is not None and hit[0] == tag and hit[2]() is W:     # the weak reference guards against a recycled id / address
        return hit[1]
    planes = ops.tc_split(W, W.shape[0], W.shape[1], W.stride(0))
    if len(_weight_planes) > 4096:
        _weight_planes.clear()
    _weight_planes[key] = (tag, planes, weakref.ref(W))
    return planes


def linear(x, W, M, m_dev=None, bias=None, epilogue=None, out=None, x_planes=None, w_planes=None, **epi):
    """out[M,N] = epi(x[M,K] @ W[N,K]^T)"""
    N, K = W.shape
    if out is None:
        out = _empty((M, N), W.device)
    if epilogue is None:
        epilogue = EPI_BIAS if bias is not None else EPI_NONE
    ops.gemm(x, W, out, M, N, K, x.stride(0) if x is not None else K, W.stride(0), out.stride(0), False, True, epilogue, bias=bias,
             m_dev=m_dev, a_planes=x_planes, b_planes=w_planes if w_planes is not None else weight_planes(W), **epi)
    return out


def matmul_nn(x, W, M, m_dev=None, out=None, x_planes=None, w_planes=None, **epi):
    """out[M,K] = x[M,N] @ W[N,K]   (dgrad of a Linear with weight W, or a fold K^T q)"""
    N, K = W.shape
    if out is None:
        out = _empty((M, K), W.device)
    ops.gemm(x, W, out, M, K, N, x.stride(0) if x is not None else x_planes.pitch, W.stride(0), out.stride(0), False, False, m_dev=m_dev,
             a_planes=x_planes, b_planes=w_planes if w_planes is not None else weight_planes(W), **epi)
    return out


def wgrad(dy, x, M, N, K, k_dev=None, out=None, accumulate=False, dy_planes=None, x_planes=None):
    """out[N,K] = dy[M,N]^T @ x[M,K]   (contraction over the M rows / tokens)"""
    if out is None:
        out = _empty((N, K), dy.device if dy is not None else dy_planes.buf.device)
    # an operand may exist only as planes (None here): its leading dimension is then only checked against the shape
    ops.gemm(dy, x, out, N, K, M, dy.stride(0) if dy is not None else dy_planes.pitch, x.stride(0) if x is not None else K,
             out.stride(0), True, False, k_dev=k_dev,
             accumulate=accumulate, a_planes=dy_planes, b_planes=x_planes)
    return out


def split_tokens(x, cap, cols, ntok, colsum_out=None):
    """hi/lo operand planes of a packed per-token tensor, shared by every GEMM that consumes it (forward,
    dgrad and wgrad read the same row-major planes; the row tail beyond the token count is zero-filled).
    ``colsum_out`` [cols]: also the column sums over the valid tokens (a bias gradient) from the same pass."""
    return ops.tc_split(x, cap, cols, x.stride(0), ntok, colsum_out=colsum_out)


def colsum(X, M, N, m_dev=None, out=None, accumulate=False):
    if out is None:
        out = _empty((N,), X.device)
    ops.colsum(X, X.stride(0), M, N, out, accumulate, m_dev)
    return out


# ------------------------------------------------------------------------------------------------
# CNE
# ------------------------------------------------------------------------------------------------
CNE_PARAM_NAMES = (
    ['word_embedding.weight', 'category_embedding.weight', 'subCategory_embedding.weight']
    + ['%s_lstm.%s_l0%s' % (x, w, s) for x in ('title', 'content') for s in ('', '_reverse')
       for w in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh')]
    + ['%s_%s' % (x, w) for x in ('title', 'content') for w in ('H.weight', 'M.weight', 'M.bias')]
    + ['%s_self_attention.%s' % (x, w) for x in ('title', 'content') for w in ('affine1.weight', 'affine1.bias', 'affine2.weight')]
)
CNE_CROSS_PARAM_NAMES = ['%s_cross_attention.%s' % (x, w) for x in ('title', 'content') for w in ('K.weight', 'Q.weight', 'Q.bias')]
CNE_GATE_PARAM_NAMES = ['%s_%s' % (x, w) for x in ('title', 'content') for w in ('H.weight', 'M.weight', 'M.bias')]


def cne_param_names(cross_attention=True, gate=True, modalities=('title', 'content')):
    """parameter order of CNEFunction for a variant: CNE (both), CNE_wo_CA (no cross attention,
    variantEncoders.py:263-339), CNE_wo_CS (no selective gate, :190-260), CNE_Title / CNE_Content (one modality,
    LSTM + self attention only, :14-99)"""
    single = len(modalities) == 1
    names = [n for n in CNE_PARAM_NAMES if (gate and not single) or n not in CNE_GATE_PARAM_NAMES]
    names += CNE_CROSS_PARAM_NAMES if (cross_attention and not single) else []
    if single:
        drop = 'content_' if modalities[0] == 'title' else 'title_'
        names = [n for n in names if not n.startswith(drop)]
    return names


class _Mod:
    """per-modality forward state"""
    pass


def _sort_desc(keys, max_key):
    """sorted indices of ``sort_fn(keys, descending=True)``.  With the default ``torch.sort`` on a CUDA tensor the
    counting-sort kernel gives the same permutation (stable, like ATen's radix sort) in one small launch."""
    if sort_fn is torch.sort and keys.is_cuda and keys.numel() <= 8192 and max_key <= 1024:
        return ops.length_sort_desc(keys.contiguous(), max_key)
    return sort_fn(keys, descending=True)[1]


def _domain_sorts(len64, domains, max_key):
    """newsEncoders.py:112-115 per pairing domain (one reference news_encoder(...) call each): the same two
    torch.sort calls on that call's lengths; indices are returned in global row numbering."""
    sorted_idx, desorted_idx = [], []
    for start, count in domains:
        si = _sort_desc(len64[start:start + count], max_key)
        # newsEncoders.py:113,115 sort the permutation again to invert it; the inverse of a permutation is
        # unique, so a scatter gives the identical result without a second radix sort
        di = torch.empty_like(si).scatter_(0, si, torch.arange(count, device=si.device))
        sorted_idx.append(si + start)
        desorted_idx.append(di)
    return sorted_idx, desorted_idx


def _cne_prepare(ids, mask_u8, N, L, domains):
    """sequence bookkeeping of one modality (newsEncoders.py:106-115): lengths, packed offsets, token -> row map, the
    per-domain sort permutations and the longest-first tile order of the recurrence.  A few small kernels."""
    dev = ids.device
    cap = N * L
    m = _Mod()
    m.L, m.cap, m.ids = L, cap, ids
    m.len = _empty((N,), dev, torch.int32)
    m.off = _empty((N + 1,), dev, torch.int32)
    m.tok_row = _empty((cap,), dev, torch.int32)
    ops.seq_prepare(mask_u8, m.len, m.off, m.tok_row)
    m.ntok = m.off[N:]                                         # device scalar (view), no sync
    # newsEncoders.py:112-115 -- same torch.sort calls (tie-breaking of the device's sort), per domain
    len64 = m.len.long()
    m.sorted_idx, m.desorted_idx = _domain_sorts(len64, domains, L)
    if len(domains) == 1:
        m.order = m.sorted_idx[0].to(torch.int32)
    else:                                                     # LSTM tiling only needs "longest first"
        m.order = _sort_desc(len64, L).to(torch.int32)
    return m


def _cne_recurrent(P, x, m, N, E, Hd, training, p_drop, seed, want_h_planes=False):
    """embedding gather + dropout, input projection, bidirectional LSTM of one modality (newsEncoders.py:117-127)"""
    dev = m.ids.device
    ids, L, cap = m.ids, m.L, m.cap
    m.seed = seed
    m.p = p_drop if training else 0.0
    table = P['word_embedding.weight']
    fused_planes = ops.default_algo() != ops.ALGO_SIMT and E % 4 == 0 and table.data_ptr() % 16 == 0
    if fused_planes:       # the embedded tokens feed GEMMs only: write them as operand planes, no fp32 [tokens, E] tensor
        m.emb = None
        m.emb_pl = ops.embed_gather_planes_fwd(table, ids, m.len, m.off, cap, m.p, seed)
    else:
        m.emb = _empty((cap, E), dev)
        ops.embed_gather_fwd(table, ids, m.len, m.off, m.emb, m.p, seed)
    pre = x + '_lstm.'
    m.w_ih = torch.cat([P[pre + 'weight_ih_l0'], P[pre + 'weight_ih_l0_reverse']], 0)          # [8H, E]
    m.w_hh = torch.stack([P[pre + 'weight_hh_l0'], P[pre + 'weight_hh_l0_reverse']], 0)        # [2, 4H, H]
    bias = torch.cat([P[pre + 'bias_ih_l0'] + P[pre + 'bias_hh_l0'],
                      P[pre + 'bias_ih_l0_reverse'] + P[pre + 'bias_hh_l0_reverse']], 0)       # [8H]
    if not fused_planes:
        m.emb_pl = split_tokens(m.emb, cap, E, m.ntok)
    m.w_ih_pl = ops.tc_split(m.w_ih, 8 * Hd, E, m.w_ih.stride(0))                              # shared with the dgrad GEMM
    m.gates = linear(m.emb, m.w_ih, cap, m.ntok, bias, x_planes=m.emb_pl, w_planes=m.w_ih_pl)  # gx, then the stash
    m.h = _empty((cap, 2 * Hd), dev)
    m.c_stash = _empty((cap, 2 * Hd), dev)
    m.c_n = _empty((N, 2 * Hd), dev)
    m.h_pl = None
    if want_h_planes and ops.lstm_fwd_planes_supported(Hd):
        # h feeds GEMMs (selective gate, two weight gradients): the recurrence writes its operand planes next to the fp32 states
        m.h_pl = ops.lstm_fwd_planes(m.gates, m.w_hh, m.len, m.off, m.order, N, L, Hd, m.h, m.c_stash, m.c_n, cap)
    else:
        ops.lstm_fwd(m.gates, m.w_hh, m.len, m.off, m.order, N, L, Hd, m.h, m.c_stash, m.c_n)
    return m


def _cne_modality_forward(P, x, ids, mask_u8, N, L, E, Hd, training, p_drop, seed, domains):
    return _cne_recurrent(P, x, _cne_prepare(ids, mask_u8, N, L, domains), N, E, Hd, training, p_drop, seed, True)


def _cne_gate_self(P, x, m, m_other_cn, partner, N, Hd, A, gate=True):
    """selective gate (newsEncoders.py:128-131) + additive self attention (:133-134); gate=False (CNE_wo_CS,
    variantEncoders.py:250-252): the attentions read the LSTM states directly"""
    dev = m.h.device
    D2 = 2 * Hd
    if gate:
        m.partner = partner
        m.cm_sel = m_other_cn.index_select(0, partner)                                            # [N, 2H]
        m.cm_sel_pl = _shared_split(m.cm_sel, N, D2)
        m.mproj = linear(m.cm_sel, P[x + '_M.weight'], N, None, P[x + '_M.bias'], x_planes=m.cm_sel_pl)   # [N, 2H]
        m.g = _empty((m.cap, D2), dev)
        if m.h_pl is None:
            m.h_pl = split_tokens(m.h, m.cap, D2, m.ntok)
        # the gated states feed the attention projection and its weight gradient: the epilogue also writes their planes
        m.hg_pl = ops.planes_empty(m.cap, D2, dev) if D2 % 8 == 0 else None
        m.hg = linear(m.h, P[x + '_H.weight'], m.cap, m.ntok, None, EPI_GATE, rowbias=m.mproj, ldrowbias=D2,
                      rowmap=m.tok_row, aux=m.h, ldaux=D2, aux_out=m.g, ldaux_out=D2, x_planes=m.h_pl, c_planes=m.hg_pl)
    else:
        m.hg = m.h
        m.hg_pl = m.h_pl
    sa = x + '_self_attention.'
    if m.hg_pl is None:
        m.hg_pl = split_tokens(m.hg, m.cap, D2, m.ntok)
    m.u = linear(m.hg, P[sa + 'affine1.weight'], m.cap, m.ntok, P[sa + 'affine1.bias'], EPI_BIAS_TANH, x_planes=m.hg_pl)
    m.self_out = _empty((N, D2), dev)
    m.alpha_self = _empty((m.cap,), dev)
    ops.attn_pool_fwd(X=m.hg, ldx=D2, D=D2, S=N, max_len=m.L, mode=0, seg_off=m.off, seg_order=m.order, U=m.u, ldu=A, A=A,
                      w2=P[sa + 'affine2.weight'], pooled=m.self_out, ldp=D2, alpha=m.alpha_self)


def _cne_cross(P, x, m, other_self, N, Hd, A):
    """cross attention (newsEncoders.py:136-137, layers.py:196-203) with K folded onto the query"""
    dev = m.h.device
    D2 = 2 * Hd
    ca = x + '_cross_attention.'
    m.other_self = other_self
    m.other_self_pl = _shared_split(other_self, N, D2)          # planes kept for the weight-gradient GEMMs of the backward
    m.q = linear(other_self, P[ca + 'Q.weight'], N, None, P[ca + 'Q.bias'], x_planes=m.other_self_pl)   # [N, A]
    m.q_pl = _shared_split(m.q, N, A)
    m.qk = matmul_nn(m.q, P[ca + 'K.weight'], N, x_planes=m.q_pl)                              # [N, 2H] = q K
    m.cross_out = _empty((N, D2), dev)
    m.alpha_cross = _empty((m.cap,), dev)
    ops.attn_pool_fwd(X=m.hg, ldx=D2, D=D2, S=N, max_len=m.L, mode=1, seg_off=m.off, seg_order=m.order, qvec=m.qk, ldq=D2,
                      scale=1.0 / math.sqrt(float(A)), pooled=m.cross_out, ldp=D2, alpha=m.alpha_cross)


class CNEFunction(torch.autograd.Function):
    """rep[N, 4H+Ec+Es] = CNE(title, content, category, subCategory); params in CNE_PARAM_NAMES order."""

    @staticmethod
    def forward(ctx, meta, title_text, title_mask, content_text, content_mask, category, subCategory, *params):
        gate = meta.get('gate', True)
        modalities = meta.get('modalities', ('title', 'content'))
        names = cne_param_names(meta['cross_attention'], gate, modalities)
        P = dict(zip(names, params))
        N, T, Lc = meta['N'], meta['T'], meta['A_len']
        E, Hd, A = meta['E'], meta['Hd'], meta['att']
        training, p = meta['training'], meta['p_drop']
        seeds = [fresh_seed() for _ in range(3)] if (training and p > 0) else [0, 0, 0]
        domains = meta.get('domains') or [(0, N)]
        if len(modalities) == 1:                      # CNE_Title / CNE_Content: LSTM -> self attention -> fusion
            x = modalities[0]
            if x == 'title':
                m = _cne_modality_forward(P, x, title_text.view(N, T), title_mask.reshape(N, T), N, T, E, Hd, training, p, seeds[0], domains)
            else:
                m = _cne_modality_forward(P, x, content_text.view(N, Lc), content_mask.reshape(N, Lc), N, Lc, E, Hd, training, p, seeds[1], domains)
            _cne_gate_self(P, x, m, None, None, N, Hd, A, False)
            cat_t, sub_t = P['category_embedding.weight'], P['subCategory_embedding.weight']
            rep = _empty((N, 2 * Hd + cat_t.shape[1] + sub_t.shape[1]), title_text.device)
            cat_i, sub_i = category.reshape(N).contiguous(), subCategory.reshape(N).contiguous()
            ops.news_fuse_fwd(m.self_out, None, None, None, cat_t, sub_t, cat_i, sub_i, N, 2 * Hd, p if training else 0.0, seeds[2], rep)
            ctx.meta, ctx.P, ctx.t, ctx.c = meta, P, (m if x == 'title' else None), (m if x == 'content' else None)
            ctx.cat_i, ctx.sub_i, ctx.fuse_seed = cat_i, sub_i, seeds[2]
            ctx.names = names
            return rep
        # title on the side lane, content on the caller's stream; joined at the exchange points
        lanes = Lanes(title_text.device)
        t, c = lanes.run(lambda: _cne_prepare(title_text.view(N, T), title_mask.reshape(N, T), N, T, domains),
                         lambda: _cne_prepare(content_text.view(N, Lc), content_mask.reshape(N, Lc), N, Lc, domains))
        lanes.fork()
        # the content branch (gather, input projection, 128-step recurrence) is the critical path of the forward stage
        _cne_recurrent(P, 'content', c, N, E, Hd, training, p, seeds[1], True)
        lanes.on_side(_cne_recurrent, P, 'title', t, N, E, Hd, training, p, seeds[0], True)
        # pairing by sort rank inside each domain (newsEncoders.py:124-129, SURVEY finding 2): title row r of a call is
        # gated with the content memory of the news at the same sorted rank.  (A handful of [N]-sized kernels: issued here
        # they run under the title branch's gather / GEMM instead of between the recurrences and the gates.)
        partner_t = torch.cat([cs.index_select(0, td) for cs, td in zip(c.sorted_idx, t.desorted_idx)])
        partner_c = torch.cat([ts.index_select(0, cd) for ts, cd in zip(t.sorted_idx, c.desorted_idx)])
        t.partner, c.partner = partner_t, partner_c
        lanes.join()
        lanes.run(lambda: _cne_gate_self(P, 'title', t, c.c_n, partner_t, N, Hd, A, gate),
                  lambda: _cne_gate_self(P, 'content', c, t.c_n, partner_c, N, Hd, A, gate))
        if meta['cross_attention']:
            lanes.run(lambda: _cne_cross(P, 'title', t, c.self_out, N, Hd, A),
                      lambda: _cne_cross(P, 'content', c, t.self_out, N, Hd, A))
        cat_t, sub_t = P['category_embedding.weight'], P['subCategory_embedding.weight']
        Dout = 4 * Hd + cat_t.shape[1] + sub_t.shape[1]
        rep = _empty((N, Dout), title_text.device)
        cat_i, sub_i = category.reshape(N).contiguous(), subCategory.reshape(N).contiguous()
        ops.news_fuse_fwd(t.self_out, t.cross_out if meta['cross_attention'] else None, c.self_out,
                          c.cross_out if meta['cross_attention'] else None, cat_t, sub_t, cat_i, sub_i, N, 2 * Hd,
                          p if training else 0.0, seeds[2], rep)
        ctx.meta, ctx.P, ctx.t, ctx.c = meta, P, t, c
        ctx.cat_i, ctx.sub_i, ctx.fuse_seed = cat_i, sub_i, seeds[2]
        ctx.names = names
        return rep

    @staticmethod
    def backward(ctx, drep):
        meta, P, t, c = ctx.meta, ctx.P, ctx.t, ctx.c
        N, E, Hd, A = meta['N'], meta['E'], meta['Hd'], meta['att']
        D2 = 2 * Hd
        dev = drep.device
        drep = drep.contiguous()
        G = {}
        modalities = meta.get('modalities', ('title', 'content'))
        single = len(modalities) == 1
        cross = meta['cross_attention'] and not single
        training, p = meta['training'], meta['p_drop']
        # 1. split + category tables (the table gradients are leaves: lane 2)
        lanes = Lanes(dev)
        d_a, d_b = _empty((N, D2), dev), (None if single else _empty((N, D2), dev))
        G['category_embedding.weight'] = _empty(P['category_embedding.weight'].shape, dev)
        G['subCategory_embedding.weight'] = _empty(P['subCategory_embedding.weight'].shape, dev)
        Ec, Es = P['category_embedding.weight'].shape[1], P['subCategory_embedding.weight'].shape[1]
        ops.news_fuse_split_bwd(drep, N, D2, Ec, Es, d_a, d_b)
        lanes.fork(2)
        lanes.on_side(ops.news_fuse_tables_bwd, drep, ctx.cat_i, ctx.sub_i, N, D2 if single else 2 * D2, p if training else 0.0,
                      ctx.fuse_seed, G['category_embedding.weight'], G['subCategory_embedding.weight'], False, lane=2)
        scale = 1.0 / math.sqrt(float(A))
        if single:
            d_self = d_out = {modalities[0]: d_a}
            mods = {modalities[0]: t if modalities[0] == 'title' else c}
        else:
            d_self = {'title': d_a, 'content': d_b}
            d_out = {'title': d_a, 'content': d_b}
            mods = {'title': t, 'content': c}
        other = {'title': 'content', 'content': 'title'}
        for x, m in mods.items():
            m.dhg = _empty((m.cap, D2), dev)
        dhg_written = {'title': False, 'content': False}
        gate = meta.get('gate', True) and not single
        wemb = P['word_embedding.weight']

        def staged(fn, *per_mod):
            """fn(x, m, ...) for every modality: title on the side lane and content on the caller's stream when both exist"""
            if single:
                x = modalities[0]
                return {x: fn(x, mods[x], *[a[x] for a in per_mod])}
            rt, rc = lanes.run(lambda: fn('title', t, *[a['title'] for a in per_mod]),
                               lambda: fn('content', c, *[a['content'] for a in per_mod]))
            return {'title': rt, 'content': rc}

        # 2. cross attention backward (produces the extra gradient of the other modality's self vector)
        def cross_bwd(x, m):
            ca = x + '_cross_attention.'
            dqk = _empty((N, D2), dev)
            ops.attn_pool_bwd(X=m.hg, ldx=D2, D=D2, S=N, max_len=m.L, mode=1, seg_off=m.off, seg_order=m.order, qvec=m.qk, ldq=D2,
                              scale=scale, alpha=m.alpha_cross, dpooled=d_out[x], lddp=D2, dX=m.dhg, lddx=D2,
                              accumulate_dx=False, dqvec=dqk, lddq=D2)
            dhg_written[x] = True
            dqk_pl = _shared_split(dqk, N, D2)                                         # dqk and dq feed two GEMMs each:
            dq = linear(dqk, P[ca + 'K.weight'], N, x_planes=dqk_pl)                      # [N,A] = dqk K^T
            G[ca + 'K.weight'] = wgrad(m.q, dqk, N, A, D2, dy_planes=m.q_pl, x_planes=dqk_pl)   # q^T dqk
            dbq = _empty((A,), dev)
            dq_pl = _shared_split(dq, N, A, colsum_out=dbq)                             # one split (+ the bias gradient)
            G[ca + 'Q.weight'] = wgrad(dq, m.other_self, N, A, D2, dy_planes=dq_pl, x_planes=m.other_self_pl)
            G[ca + 'Q.bias'] = dbq
            # d(other self) = dq Q + its own output gradient
            return matmul_nn(dq, P[ca + 'Q.weight'], N, epilogue=EPI_ADD_AUX, aux=d_out[other[x]], ldaux=D2, x_planes=dq_pl)

        if cross:
            r = staged(cross_bwd)
            d_self = {'content': r['title'], 'title': r['content']}

        # 3. self attention backward, 4. selective gate backward
        def self_gate_bwd(x, m, d_self_x):
            sa = x + '_self_attention.'
            dU = _empty((m.cap, A), dev)
            dw2p = _empty((N, A), dev)
            ops.attn_pool_bwd(X=m.hg, ldx=D2, D=D2, S=N, max_len=m.L, mode=0, seg_off=m.off, seg_order=m.order, U=m.u, ldu=A, A=A,
                              w2=P[sa + 'affine2.weight'], alpha=m.alpha_self, dpooled=d_self_x, lddp=D2, dX=m.dhg,
                              lddx=D2, accumulate_dx=dhg_written[x], dU=dU, lddu=A, dw2_partial=dw2p)
            G[sa + 'affine2.weight'] = colsum(dw2p, N, A).view(1, A)
            db1 = _empty((A,), dev)
            dU_pl = split_tokens(dU, m.cap, A, m.ntok, colsum_out=db1)
            matmul_nn(dU, P[sa + 'affine1.weight'], m.cap, m.ntok, out=m.dhg, accumulate=True, x_planes=dU_pl)
            # (weight gradients are leaves: lane 2, under the memory-bound gate backward and the next data-gradient GEMM)
            G[sa + 'affine1.weight'] = lanes.leaf(wgrad, dU, m.hg, m.cap, A, D2, k_dev=m.ntok, dy_planes=dU_pl, x_planes=m.hg_pl)
            G[sa + 'affine1.bias'] = db1
            lanes.keep.extend((dU, dU_pl, m.hg_pl))   # released at the join: a lane never hands memory back while another may read it
            m.hg_pl = None
            if not gate:                       # CNE_wo_CS / single modality: hg is h, nothing flows into another cell state
                m.dh = m.dhg
                return None
            dh0 = _empty((m.cap, D2), dev)
            dmproj = _empty((N, D2), dev)
            if ops.default_algo() != ops.ALGO_SIMT:
                # dz only feeds the two GEMMs below and the per-news sum: one pass writes its planes, dmproj and dh0
                dz = None
                dz_pl = ops.gate_bwd_planes(m.dhg, m.h, m.g, m.off, N, D2, m.cap, dh0, dmproj)
            else:
                dz = _empty((m.cap, D2), dev)
                ops.gate_bwd_pre(m.dhg, m.h, m.g, m.cap * D2, m.ntok, D2, dz, dh0)
                dz_pl = split_tokens(dz, m.cap, D2, m.ntok)
                ops.segment_colsum(dz, D2, m.off, N, D2, dmproj, D2)
            m.dh = matmul_nn(dz, P[x + '_H.weight'], m.cap, m.ntok, epilogue=EPI_ADD_AUX, aux=dh0, ldaux=D2, out=m.dhg,
                             x_planes=dz_pl)
            G[x + '_H.weight'] = lanes.leaf(wgrad, dz, m.h, m.cap, D2, D2, k_dev=m.ntok, dy_planes=dz_pl, x_planes=m.h_pl)
            lanes.keep.extend((m.h_pl, dz, dz_pl))
            m.h_pl = None
            dbm = _empty((D2,), dev)
            dmproj_pl = _shared_split(dmproj, N, D2, colsum_out=dbm)                       # shared by both GEMMs, + bias gradient
            G[x + '_M.weight'] = wgrad(dmproj, m.cm_sel, N, D2, D2, dy_planes=dmproj_pl, x_planes=m.cm_sel_pl)
            G[x + '_M.bias'] = dbm
            return matmul_nn(dmproj, P[x + '_M.weight'], N, x_planes=dmproj_pl)               # grad of cn_other[partner]

        d_cm_sel = staged(self_gate_bwd, d_self)
        # partner_t and partner_c are inverse permutations of each other
        if gate:
            dcn = {'content': d_cm_sel['title'].index_select(0, c.partner),
                   'title': d_cm_sel['content'].index_select(0, t.partner)}
        else:
            dcn = {x: torch.zeros(N, D2, device=dev) for x in mods}

        # 5. LSTM backward, input projection, embedding scatter.  Per modality: the recurrence, then the data gradient of the
        # input projection and its scatter into the word table, then the weight gradients (leaves).  The two scatters add
        # into the same table in a fixed order (title, content), so both go to lane 1; the content branch's weight-gradient
        # GEMMs -- the bulk of what is left -- run on the caller's stream meanwhile.
        # With a flat gradient buffer (trainer.TrainStep) the scatter adds straight into the table's .grad view: no [V, E]
        # temporary, no memset of it, no [V, E] add afterwards.
        in_place = _flat_grads(P, ctx.names) and wemb.grad.is_contiguous() and wemb.grad.data_ptr() % 16 == 0
        dtable = wemb.grad if in_place else _empty(wemb.shape, dev)
        first = [not in_place]

        def recurrence_bwd(x, m, dcn_x):
            db = _empty((8 * Hd,), dev)
            if m.emb is None and ops.lstm_bwd_planes_supported(Hd):
                # dL/dgx only feeds GEMMs and the bias gradient: the recurrence writes its operand planes and column sums
                dz = None
                dz_pl = ops.lstm_bwd_planes(m.gates, m.c_stash, m.w_hh, m.len, m.off, m.order, N, m.L, Hd, m.dh,
                                            dcn_x.contiguous(), m.cap, db)
            else:
                ops.lstm_bwd(m.gates, m.c_stash, m.w_hh, m.len, m.off, m.order, N, m.L, Hd, m.dh, dcn_x.contiguous())
                dz = m.gates                                                                  # [cap, 8H] = dL/dgx
                dz_pl = split_tokens(dz, m.cap, 8 * Hd, m.ntok, colsum_out=db)
            demb = matmul_nn(dz, m.w_ih, m.cap, m.ntok, x_planes=dz_pl, w_planes=m.w_ih_pl)
            return dz, dz_pl, db, demb

        def scatter(x, m, demb):
            ops.embed_gather_bwd(demb, m.ids, m.len, m.off, dtable, m.p, m.seed, not first[0])
            first[0] = False

        def shifted_h(m, planes):
            """h_{t-1} of every token = the second operand of the recurrent weight gradient; a GEMM operand only: straight to planes"""
            if planes:
                return None, ops.lstm_shift_h_planes(m.h, m.len, m.off, m.tok_row, N, m.L, Hd, m.cap)
            hprev = _empty((m.cap, D2), dev)
            ops.lstm_shift_h(m.h, m.len, m.off, m.tok_row, N, m.L, Hd, hprev)
            return hprev, None

        def weight_grads(x, m, dz, dz_pl, db, hp=None):
            pre = x + '_lstm.'
            # as 16-bit planes the reverse half of h_{t-1} starts at column Hd, 16 B aligned only when Hd % 8 == 0: otherwise fp32
            hprev, hprev_pl = hp if hp is not None else shifted_h(m, dz_pl is not None and Hd % 8 == 0)
            for d, sfx in enumerate(('', '_reverse')):
                G[pre + 'weight_hh_l0' + sfx] = wgrad(dz[:, d * 4 * Hd:(d + 1) * 4 * Hd] if dz is not None else None,
                                                     hprev[:, d * Hd:(d + 1) * Hd] if hprev is not None else None,
                                                     m.cap, 4 * Hd, Hd, k_dev=m.ntok,
                                                     dy_planes=dz_pl.cols(d * 4 * Hd, (d + 1) * 4 * Hd) if dz_pl else None,
                                                     x_planes=hprev_pl.cols(d * Hd, (d + 1) * Hd) if hprev_pl else None)
            dwih = wgrad(dz, m.emb, m.cap, 8 * Hd, E, k_dev=m.ntok, dy_planes=dz_pl, x_planes=m.emb_pl)
            lanes.keep.extend((m.emb_pl, hprev, hprev_pl))
            m.emb_pl = None
            for d, sfx in enumerate(('', '_reverse')):
                G[pre + 'weight_ih_l0' + sfx] = dwih[d * 4 * Hd:(d + 1) * 4 * Hd]
                G[pre + 'bias_ih_l0' + sfx] = db[d * 4 * Hd:(d + 1) * 4 * Hd]
                G[pre + 'bias_hh_l0' + sfx] = db[d * 4 * Hd:(d + 1) * 4 * Hd]

        if single:
            x = modalities[0]
            dz, dz_pl, db, demb = recurrence_bwd(x, mods[x], dcn[x])
            scatter(x, mods[x], demb)
            weight_grads(x, mods[x], dz, dz_pl, db)
        else:
            # lane 1: title recurrence, title scatter, content scatter (the chain the end of the backward pass waits for);
            # lane 2: the title branch's weight gradients; caller's stream: content recurrence, content weight gradients
            lanes.fork()
            # the content recurrence must get the SMs first -- its longest sequences are the critical path of this stage
            # and the title recurrence fits into the SMs its short tiles leave idle: the title lane starts with a kernel
            # it needs anyway (h_{t-1} planes), so its recurrence is launched a few microseconds after the content one
            planes = t.emb is None and ops.lstm_bwd_planes_supported(Hd)
            thp = lanes.on_side(shifted_h, t, planes)
            dz, dz_pl, db, demb = recurrence_bwd('content', c, dcn['content'])
            tz, tz_pl, tdb, tdemb = lanes.on_side(recurrence_bwd, 'title', t, dcn['title'])
            lanes.on_side(scatter, 'title', t, tdemb)
            lanes.fork(2, after=1)
            lanes.on_side(weight_grads, 'title', t, tz, tz_pl, tdb, thp, lane=2)
            lanes.keep.extend((tz, tz_pl, tdemb, dz, dz_pl, demb, thp))
            lanes.fork()                                       # lane 1, behind the title scatter
            lanes.on_side(scatter, 'content', c, demb)
            if in_place:
                lanes.on_side(_notify, 'table')               # the table gradient is final once lane 1 gets here
            weight_grads('content', c, dz, dz_pl, db)
        lanes.join()
        G['word_embedding.weight'] = None if in_place else dtable
        ctx.t = ctx.c = None
        pg = _param_grads(P, ctx.names, G)
        if in_place:
            _notify('cne')
            if single:
                _notify('table')
        return (None,) * 7 + pg


# ------------------------------------------------------------------------------------------------
# SUE
# ------------------------------------------------------------------------------------------------
def _gcn_param_names(L, layer_norm=False):
    names = []
    for l in range(L):
        names += ['gcn.gcn_layers.%d.W.weight' % l, 'gcn.gcn_layers.%d.W.bias' % l]
        if layer_norm:                                    # layers.py:274-275
            names += ['gcn.gcn_layers.%d.layer_normalization.weight' % l, 'gcn.gcn_layers.%d.layer_normalization.bias' % l]
    return names


def sue_param_names(L, layer_norm=False):
    return (['proxy_node_embedding'] + _gcn_param_names(L, layer_norm)
            + ['intraCluster_K.weight', 'intraCluster_Q.weight', 'intraCluster_Q.bias', 'clusterFeatureAffine.weight',
               'clusterFeatureAffine.bias', 'interClusterAttention.K.weight', 'interClusterAttention.Q.weight',
               'interClusterAttention.Q.bias'])


def sue_wo_gcn_param_names():
    """SUE_wo_GCN (variantEncoders.py:342-390): no proxy nodes / GCN; intraCluster_K has a bias there"""
    return ['intraCluster_K.weight', 'intraCluster_K.bias', 'intraCluster_Q.weight', 'intraCluster_Q.bias',
            'clusterFeatureAffine.weight', 'clusterFeatureAffine.bias', 'interClusterAttention.K.weight',
            'interClusterAttention.Q.weight', 'interClusterAttention.Q.bias']


def sue_wo_hca_param_names(L, layer_norm=False):
    return (['proxy_node_embedding'] + _gcn_param_names(L, layer_norm)
            + ['attention.affine1.weight', 'attention.affine1.bias', 'attention.affine2.weight'])


def sue_names(meta):
    """parameter order of SUEFunction for the user encoder described by ``meta`` (SUE, SUE_wo_HCA, SUE_wo_GCN)"""
    gcn, ln = meta.get('gcn', True), meta.get('layer_norm', False)
    L = meta['gcn_layers'] if gcn else 0
    return (sue_param_names(L, ln) if meta['hca'] else sue_wo_hca_param_names(L, ln)) if gcn else sue_wo_gcn_param_names()


class SUEFunction(torch.autograd.Function):
    """user[B,n,D] = SUE(history_embedding[B,H,D], candidate[B,n,D], graph, cluster mask / indices)."""

    @staticmethod
    def forward(ctx, meta, hist, cand, graph, cmask, cidx, *params):
        hca = meta['hca']
        gcn = meta.get('gcn', True)
        L = meta['gcn_layers'] if gcn else 0
        names = sue_names(meta)
        P = dict(zip(names, params))
        B, H, D = hist.shape
        n = cand.shape[1]
        C = P['proxy_node_embedding'].shape[0] if gcn else meta['category_num']
        Gn, C1 = H + C, C + 1
        dev = hist.device
        training, p = meta['training'], meta['p_drop']
        pe = p if training else 0.0
        seeds = [fresh_seed() for _ in range(L + 2)] if pe > 0 else [0] * (L + 2)
        hist = hist.contiguous()
        cand = cand.contiguous()
        if not gcn:                                                                           # SUE_wo_GCN: clusters over the raw history
            return SUEFunction._clusters_forward(ctx, meta, P, names, hist, cand, cmask, cidx, seeds, (B, H, D, n, C, Gn, C1), L, pe)
        # the candidate-side projections of the cluster attentions do not depend on the GCN: side lane, joined before the
        # intra-cluster attention needs them
        lanes = Lanes(dev)
        pre = None
        if hca:
            lanes.fork()
            pre = lanes.on_side(SUEFunction._cand_side, P, cand, B, n, D)
        gfeat, graph, xs, rs, aggs, lns = SUEFunction._gcn(meta, P, hist, graph, seeds, L, pe)
        ctx.meta, ctx.P, ctx.names = meta, P, names
        ctx.dims = (B, H, D, n, C, Gn, C1)
        ctx.seeds, ctx.graph = seeds, graph
        ctx.xs, ctx.rs, ctx.aggs, ctx.lns = xs, rs, aggs, lns
        ctx.gfeat, ctx.cand = gfeat, cand
        if not hca:                                                                           # SUE_wo_HCA
            pooled, ctx.u, ctx.alpha = SUEFunction._history_pool(P, gfeat)
            return pooled.unsqueeze(1).repeat(1, n, 1)
        lanes.join()
        return SUEFunction._clusters_tail(ctx, P, gfeat, cand, cmask, cidx, seeds, (B, H, D, n, C, Gn, C1), L, pe, pre)

    @staticmethod
    def _gcn(meta, P, hist, graph, seeds, L, pe):
        """X0 = [history | proxy nodes] through the GCN layers; returns gfeat [B, H, D] = (X_L + X0)[:, :H], the contiguous
        graph and the stash of the backward pass (xs, rs, aggs, lns)"""
        B, H, D = hist.shape
        Gn = H + P['proxy_node_embedding'].shape[0]
        dev = hist.device
        residual, ln = meta['residual'], meta.get('layer_norm', False)
        # X0 = [history | dropout_(proxy nodes)]   (userEncoders.py:80)
        x0 = _empty((B, Gn, D), dev)
        x0[:, :H] = hist
        proxy = P['proxy_node_embedding'].unsqueeze(0).expand(B, -1, -1).contiguous()
        if pe > 0:
            ops.dropout(proxy, pe, seeds[L], proxy)
        x0[:, H:] = proxy
        # dense graph -> neighbour lists (and of the transpose for the backward pass)
        graph = graph.contiguous()
        nnz, col, val = _empty((B * Gn,), dev, torch.int32), _empty((B * Gn, Gn), dev, torch.int32), _empty((B * Gn, Gn), dev)
        ops.graph_to_csr(graph, False, nnz, col, val)
        # GCN layers: X <- drop(relu(W (A X) + b) + X)   (layers.py:285-292,318-323)
        xs, rs, aggs, lns = [x0], [], [], []
        x = x0
        for l in range(L):
            agg = _empty((B * Gn, D), dev)
            ops.gcn_aggregate(nnz, col, val, x, B, Gn, D, agg)
            r = _empty((B * Gn, D), dev)
            xv = x.view(B * Gn, D)
            pl = (pe / 2.0) if l < L - 1 else 0.0
            agg_pl = ops.tc_split(agg, B * Gn, D, D)             # shared with the weight-gradient GEMM of the backward
            if ln:                                                # layers.py:286-292 with layer_norm: relu(LN(W(AX)+b)) + X
                lnp = 'gcn.gcn_layers.%d.layer_normalization.' % l
                y = linear(agg, P['gcn.gcn_layers.%d.W.weight' % l], B * Gn, None, P['gcn.gcn_layers.%d.W.bias' % l], EPI_BIAS,
                           x_planes=agg_pl)
                xn = _empty((B * Gn, D), dev)
                mu, rstd = _empty((B * Gn,), dev), _empty((B * Gn,), dev)
                ops.ln_relu_res_fwd(y, P[lnp + 'weight'], P[lnp + 'bias'], xv if residual else None, B * Gn, D, 1e-5, pl, seeds[l],
                                    xn, r, mu, rstd)
                lns.append((y, mu, rstd))
            else:
                xn = linear(agg, P['gcn.gcn_layers.%d.W.weight' % l], B * Gn, None, P['gcn.gcn_layers.%d.W.bias' % l],
                            EPI_BIAS_RELU_RES, aux=xv if residual else None, ldaux=D, aux_out=r, ldaux_out=D, p_drop=pl,
                            seed=seeds[l], x_planes=agg_pl)
            aggs.append((agg, agg_pl))
            rs.append(r)
            x = xn.view(B, Gn, D)
            xs.append(x)
        gfeat = (x + x0)[:, :H, :].contiguous()                                              # userEncoders.py:81-82
        return gfeat, graph, xs, rs, aggs, lns

    @staticmethod
    def _history_pool(P, gfeat):
        """SUE_wo_HCA: additive attention over the history rows (variantEncoders.py:416-419); returns (pooled [B, D], the
        attention projection u, the weights alpha)"""
        B, H, D = gfeat.shape
        A = P['attention.affine1.weight'].shape[0]
        u = linear(gfeat.view(B * H, D), P['attention.affine1.weight'], B * H, None, P['attention.affine1.bias'], EPI_BIAS_TANH)
        pooled = _empty((B, D), gfeat.device)
        alpha = _empty((B * H,), gfeat.device)
        ops.attn_pool_fwd(X=gfeat, ldx=D, D=D, S=B, max_len=H, mode=0, fixed_len=H, U=u, ldu=A, A=A,
                          w2=P['attention.affine2.weight'], pooled=pooled, ldp=D, alpha=alpha)
        return pooled, u, alpha

    @staticmethod
    def _cand_side(P, cand, B, n, D, m_dev=None):
        """what the cluster attentions need from the candidates alone (userEncoders.py:84,94: the two query projections;
        the inter-cluster K is folded onto its query).  ``m_dev``: an int32 device scalar; only the first *m_dev of the
        B * n rows are computed (the rest of the outputs is left unwritten)"""
        Au = P['intraCluster_K.weight'].shape[0]
        cand_pl = _shared_split(cand.view(B * n, D), B * n, D, m_dev=m_dev)   # also the weight-gradient operand of the backward
        Qp = linear(cand.view(B * n, D), P['intraCluster_Q.weight'], B * n, m_dev, P['intraCluster_Q.bias'], x_planes=cand_pl)
        q2 = linear(cand.view(B * n, D), P['interClusterAttention.Q.weight'], B * n, m_dev, P['interClusterAttention.Q.bias'],
                    x_planes=cand_pl)
        q2_pl = _shared_split(q2, B * n, Au, m_dev=m_dev)
        qk2 = matmul_nn(q2, P['interClusterAttention.K.weight'], B * n, m_dev, x_planes=q2_pl)
        return cand_pl, Qp, q2, q2_pl, qk2

    @staticmethod
    def _clusters_forward(ctx, meta, P, names, hist, cand, cmask, cidx, seeds, dims, L, pe):
        ctx.meta, ctx.P, ctx.names = meta, P, names
        ctx.dims = dims
        ctx.seeds, ctx.graph = seeds, None
        ctx.xs, ctx.rs, ctx.aggs = None, None, None
        ctx.gfeat, ctx.cand = hist, cand
        return SUEFunction._clusters_tail(ctx, P, hist, cand, cmask, cidx, seeds, dims, L, pe)

    @staticmethod
    def _user_keys(P, gfeat):
        """what the cluster attentions need from the history alone: gfeat's operand planes and the keys of the intra-cluster
        attention (userEncoders.py:85)"""
        B, H, D = gfeat.shape
        gfeat_pl = _shared_split(gfeat.view(B * H, D), B * H, D)   # gfeat, cand, q2: split once for the forward GEMMs and the
        Kp = linear(gfeat.view(B * H, D), P['intraCluster_K.weight'], B * H, x_planes=gfeat_pl)   # weight-gradient GEMMs of the backward
        return gfeat_pl, Kp

    @staticmethod
    def _clusters_tail(ctx, P, gfeat, cand, cmask, cidx, seeds, dims, L, pe, pre=None, keys=None):
        """intra-cluster attention, cluster affine, inter-cluster attention (userEncoders.py:83-97); ``keys``: the result of
        _user_keys when the history side is already computed"""
        B, H, D, n, C, Gn, C1 = dims
        dev = gfeat.device
        Au = P['intraCluster_K.weight'].shape[0]
        scale = 1.0 / math.sqrt(float(Au))
        # (an intraCluster_K.bias -- SUE_wo_GCN only -- shifts every score of a (user, candidate) pair equally and
        #  cancels in the per-cluster softmax: it is not applied, and its gradient is exactly zero)
        cand_pl, Qp, q2, q2_pl, qk2 = pre if pre is not None else SUEFunction._cand_side(P, cand, B, n, D)
        gfeat_pl, Kp = keys if keys is not None else SUEFunction._user_keys(P, gfeat)
        alpha = _empty((B * n, H), dev)
        intra = _empty((B * n * C1, D), dev)
        cidx = cidx.contiguous()
        ops.cluster_intra_fwd(Kp, Qp, gfeat, cidx, B, n, H, Au, D, C1, scale, alpha, intra)
        r_f = _empty((B * n * C1, D), dev)
        intra_pl = ops.tc_split(intra, B * n * C1, D, D)         # shared with the weight-gradient GEMM of the backward
        f = linear(intra, P['clusterFeatureAffine.weight'], B * n * C1, None, P['clusterFeatureAffine.bias'],
                   EPI_BIAS_RELU_RES, aux=intra, ldaux=D, aux_out=r_f, ldaux_out=D, p_drop=pe, seed=seeds[L + 1],
                   x_planes=intra_pl)
        cm = cmask.unsqueeze(1).expand(-1, n, -1).contiguous().view(torch.uint8)             # [B,n,C1]
        user = _empty((B * n, D), dev)
        alpha2 = _empty((B * n * C1,), dev)
        ops.attn_pool_fwd(X=f, ldx=D, D=D, S=B * n, max_len=C1, mode=1, fixed_len=C1, qvec=qk2, ldq=D, scale=scale,
                          mask=cm, pooled=user, ldp=D, alpha=alpha2)
        ctx.sv = (Kp, Qp, alpha, intra, r_f, f, q2, qk2, cm, alpha2, cidx, Au, scale, intra_pl, (gfeat_pl, cand_pl, q2_pl))
        return user.view(B, n, D)


    @staticmethod
    def backward(ctx, duser):
        meta, P = ctx.meta, ctx.P
        B, H, D, n, C, Gn, C1 = ctx.dims
        L = meta['gcn_layers'] if meta.get('gcn', True) else 0
        dev = duser.device
        G = {}
        training, p = meta['training'], meta['p_drop']
        pe = p if training else 0.0
        seeds = ctx.seeds
        gfeat, cand = ctx.gfeat, ctx.cand
        dcand = None
        lanes = Lanes(dev)

        def side_wgrad(name, dy, x, M, N_, K_, dy_pl, x_pl):
            """a weight-gradient GEMM is a leaf of the backward pass: side lane, while the caller's stream goes on with the
            chain towards the inputs (its operands stay alive until the join)"""
            lanes.keep.extend((dy, x, dy_pl, x_pl))
            lanes.fork()
            G[name] = lanes.on_side(wgrad, dy, x, M, N_, K_, dy_planes=dy_pl, x_planes=x_pl)

        if not meta['hca']:
            A = P['attention.affine1.weight'].shape[0]
            dpooled = duser.sum(dim=1).contiguous()                                          # repeat over candidates
            dg = _empty((B * H, D), dev)
            dU = _empty((B * H, A), dev)
            dw2p = _empty((B, A), dev)
            ops.attn_pool_bwd(X=gfeat, ldx=D, D=D, S=B, max_len=H, mode=0, fixed_len=H, U=ctx.u, ldu=A, A=A,
                              w2=P['attention.affine2.weight'], alpha=ctx.alpha, dpooled=dpooled, lddp=D, dX=dg, lddx=D,
                              accumulate_dx=False, dU=dU, lddu=A, dw2_partial=dw2p)
            G['attention.affine2.weight'] = colsum(dw2p, B, A).view(1, A)
            matmul_nn(dU, P['attention.affine1.weight'], B * H, out=dg, accumulate=True)
            G['attention.affine1.weight'] = wgrad(dU, gfeat.view(B * H, D), B * H, A, D)
            G['attention.affine1.bias'] = colsum(dU, B * H, A)
        else:
            Kp, Qp, alpha, intra, r_f, f, q2, qk2, cm, alpha2, cidx, Au, scale, intra_pl, (gfeat_pl, cand_pl, q2_pl) = ctx.sv
            duser = duser.contiguous().view(B * n, D)
            # inter-cluster attention backward
            df = _empty((B * n * C1, D), dev)
            dqk2 = _empty((B * n, D), dev)
            ops.attn_pool_bwd(X=f, ldx=D, D=D, S=B * n, max_len=C1, mode=1, fixed_len=C1, qvec=qk2, ldq=D, scale=scale,
                              mask=cm, alpha=alpha2, dpooled=duser, lddp=D, dX=df, lddx=D, accumulate_dx=False,
                              dqvec=dqk2, lddq=D)
            cand2 = cand.view(B * n, D)

            # side lane: everything that only leads to weight gradients and to the candidates' gradient (the query chain of
            # the inter-cluster attention, every weight-gradient GEMM); the caller's stream keeps the chain that leads to
            # the history gradient.  Joined once, before the gradients are handed to autograd.
            def query_chain():
                dqk2_pl = _shared_split(dqk2, B * n, D)                                        # operands used by two GEMMs: one split
                dq2 = linear(dqk2, P['interClusterAttention.K.weight'], B * n, x_planes=dqk2_pl)  # [B*n, Au]
                G['interClusterAttention.K.weight'] = wgrad(q2, dqk2, B * n, Au, D, dy_planes=q2_pl, x_planes=dqk2_pl)
                dbq2 = _empty((Au,), dev)
                dq2_pl = _shared_split(dq2, B * n, Au, colsum_out=dbq2)
                G['interClusterAttention.Q.weight'] = wgrad(dq2, cand2, B * n, Au, D, dy_planes=dq2_pl, x_planes=cand_pl)
                G['interClusterAttention.Q.bias'] = dbq2
                return matmul_nn(dq2, P['interClusterAttention.Q.weight'], B * n, x_planes=dq2_pl)   # [B*n, D]
            lanes.keep.append(dqk2)
            lanes.fork()
            dcand = lanes.on_side(query_chain)
            # cluster affine backward: f = (relu(W intra + b) + intra) * drop
            db_f = _empty((D,), dev)
            if _fused_relu_bwd(df, D):
                # dropout mask, relu mask, operand planes and the bias gradient in one pass over df
                df_d = _empty(df.shape, dev) if pe > 0 else None
                dpre = None
                dpre_pl = ops.relu_bwd_split_colsum(df, r_f, B * n * C1, D, pe, seeds[L + 1], df_d, db_f)
                df = df_d if pe > 0 else df
            else:
                if pe > 0:
                    ops.dropout(df, pe, seeds[L + 1], df)
                dpre = df * (r_f > 0)                                                         # relu mask
                dpre_pl = ops.tc_split(dpre, B * n * C1, D, D, colsum_out=db_f)  # planes + bias gradient in one pass
            side_wgrad('clusterFeatureAffine.weight', dpre, intra, B * n * C1, D, D, dpre_pl, intra_pl)
            G['clusterFeatureAffine.bias'] = db_f
            dintra = matmul_nn(dpre, P['clusterFeatureAffine.weight'], B * n * C1, epilogue=EPI_ADD_AUX, aux=df, ldaux=D,
                               x_planes=dpre_pl)
            # intra-cluster attention backward
            da_ws = _empty((B * n, H), dev)
            dKp, dQp = _empty((B * H, Au), dev), _empty((B * n, Au), dev)
            dg = _empty((B * H, D), dev)
            ops.cluster_intra_bwd(dintra, Kp, Qp, gfeat, cidx, alpha, B, n, H, Au, D, C1, scale, da_ws, dKp, dQp, dg, False)
            dKp_pl = _shared_split(dKp, B * H, Au)
            side_wgrad('intraCluster_K.weight', dKp, gfeat.view(B * H, D), B * H, Au, D, dKp_pl, gfeat_pl)
            matmul_nn(dKp, P['intraCluster_K.weight'], B * H, out=dg, accumulate=True, x_planes=dKp_pl)

            def cand_tail():
                dbq = _empty((Au,), dev)
                dQp_pl = _shared_split(dQp, B * n, Au, colsum_out=dbq)
                G['intraCluster_Q.weight'] = wgrad(dQp, cand2, B * n, Au, D, dy_planes=dQp_pl, x_planes=cand_pl)
                G['intraCluster_Q.bias'] = dbq
                matmul_nn(dQp, P['intraCluster_Q.weight'], B * n, out=dcand, accumulate=True, x_planes=dQp_pl)
            lanes.keep.append(dQp)
            lanes.fork()
            lanes.on_side(cand_tail)
        if not meta.get('gcn', True):                  # SUE_wo_GCN: gfeat is the history embedding itself
            G['intraCluster_K.bias'] = torch.zeros_like(P['intraCluster_K.bias'])
            lanes.join()
            ctx.sv = None
            pg = _param_grads(P, ctx.names, G)
            _notify('sue')
            return (None, dg.view(B, H, D), dcand.view(B, n, D), None, None, None) + pg
        # GCN backward.  gfeat = (x_L + x0)[:, :H]
        dxL = torch.zeros((B, Gn, D), device=dev)
        dxL[:, :H] = dg.view(B, H, D)
        dx0 = dxL.clone()
        nnzT, colT, valT = _empty((B * Gn,), dev, torch.int32), _empty((B * Gn, Gn), dev, torch.int32), _empty((B * Gn, Gn), dev)
        ops.graph_to_csr(ctx.graph, True, nnzT, colT, valT)
        dx = dxL.view(B * Gn, D)
        residual = meta['residual']
        for l in range(L - 1, -1, -1):
            pl = (pe / 2.0) if l < L - 1 else 0.0
            db_l = _empty((D,), dev)
            if meta.get('layer_norm', False):
                lnp = 'gcn.gcn_layers.%d.layer_normalization.' % l
                y, mu, rstd = ctx.lns[l]
                dx_d = _empty(dx.shape, dev) if pl > 0 else None
                dpre = _empty((B * Gn, D), dev)                   # dL/dy (pre-normalisation)
                G[lnp + 'weight'], G[lnp + 'bias'] = _empty((D,), dev), _empty((D,), dev)
                ops.ln_relu_res_bwd(dx, y, P[lnp + 'weight'], ctx.rs[l], mu, rstd, B * Gn, D, pl, seeds[l], dx_d, dpre,
                                    G[lnp + 'weight'], G[lnp + 'bias'])
                dx = dx_d if pl > 0 else dx
                dpre_pl = ops.tc_split(dpre, B * Gn, D, D, colsum_out=db_l)
            elif _fused_relu_bwd(dx, D):
                dx_d = _empty(dx.shape, dev) if pl > 0 else None
                dpre = None
                dpre_pl = ops.relu_bwd_split_colsum(dx, ctx.rs[l], B * Gn, D, pl, seeds[l], dx_d, db_l)
                dx = dx_d if pl > 0 else dx
            else:
                if pl > 0:
                    dx = dx.clone() if dx.data_ptr() == dxL.data_ptr() else dx
                    ops.dropout(dx, pl, seeds[l], dx)
                dpre = dx * (ctx.rs[l] > 0)
                dpre_pl = ops.tc_split(dpre, B * Gn, D, D, colsum_out=db_l)   # one split for the wgrad and the dgrad GEMM, + bias gradient
            side_wgrad('gcn.gcn_layers.%d.W.weight' % l, dpre, ctx.aggs[l][0], B * Gn, D, D, dpre_pl, ctx.aggs[l][1])
            G['gcn.gcn_layers.%d.W.bias' % l] = db_l
            dagg = matmul_nn(dpre, P['gcn.gcn_layers.%d.W.weight' % l], B * Gn, x_planes=dpre_pl)
            dprev = _empty((B * Gn, D), dev)
            ops.gcn_aggregate(nnzT, colT, valT, dagg, B, Gn, D, dprev, add=dx if residual else None)   # + residual term
            dx = dprev
        dx0 = dx0.view(B * Gn, D) + dx
        dx0 = dx0.view(B, Gn, D)
        dhist = dx0[:, :H].contiguous()
        dproxy_b = dx0[:, H:].contiguous()
        if pe > 0:
            ops.dropout(dproxy_b, pe, seeds[L], dproxy_b)
        G['proxy_node_embedding'] = dproxy_b.sum(dim=0)
        lanes.join()
        ctx.xs = ctx.rs = ctx.aggs = ctx.sv = ctx.lns = None
        pg = _param_grads(P, ctx.names, G)
        _notify('sue')
        return (None, dhist, dcand.view(B, n, D) if dcand is not None else None, None, None, None) + pg


class RowDot(torch.autograd.Function):
    """logits[b,k] = sum_d user[b,k,d] * news[b,k,d]   (model.py:127)"""

    @staticmethod
    def forward(ctx, user, news):
        B, n, D = user.shape
        user, news = user.contiguous(), news.contiguous()
        out = _empty((B, n), user.device)
        ops.rowdot_fwd(user, news, B * n, D, out)
        ctx.save_for_backward(user, news)
        return out

    @staticmethod
    def backward(ctx, dout):
        user, news = ctx.saved_tensors
        B, n, D = user.shape
        du, dn = torch.empty_like(user), torch.empty_like(news)
        ops.rowdot_bwd(dout.contiguous(), user, news, B * n, D, du, False, dn, False)
        return du, dn


# ------------------------------------------------------------------------------------------------
# SUE inference in two halves: the user side once per batch of users, the candidate tail per tile of candidates
# ------------------------------------------------------------------------------------------------
# Scoring a pool of candidates against the same users (news recommendation) repeats only the candidate tail of
# SUEFunction.forward: the GCN and the intra-cluster keys depend on the history alone.  Both halves call the forward's own
# pieces on the same shapes, so a tile's scores equal SUEFunction.forward + RowDot on [B, T] candidates bit for bit.
# Inference only: eval mode (no dropout), no autograd.
@torch.no_grad()
def sue_user_side(meta, hist, graph, cmask, cidx, *params, factored=False):
    """the history half of SUEFunction.forward for the users of hist [B, H, D]: returns the tuple of tensors
    ``sue_tile_scores`` takes -- (gfeat, Kp, cmask, cidx) with the hierarchical cluster attention, (pooled user vector
    [B, D], its attention weights over the history [B, H]) for SUE_wo_HCA.  ``factored``: the cluster attention's tuple
    also carries Wg = gfeat clusterFeatureAffine.weight^T [B, H, D] (no bias), for ``sue_tile_scores_factored``"""
    assert not meta['training'], 'the split SUE forward is for inference (eval mode)'
    P = dict(zip(sue_names(meta), params))
    gcn = meta.get('gcn', True)
    L = meta['gcn_layers'] if gcn else 0
    hist = hist.contiguous()
    gfeat = SUEFunction._gcn(meta, P, hist, graph, [0] * (L + 2), L, 0.0)[0] if gcn else hist
    if not meta['hca']:
        pooled, _, alpha = SUEFunction._history_pool(P, gfeat)
        return pooled, alpha.view(gfeat.shape[0], gfeat.shape[1])
    gfeat_pl, Kp = SUEFunction._user_keys(P, gfeat)
    if not factored:
        return gfeat, Kp, cmask, cidx.contiguous()
    B, H, D = gfeat.shape
    Wg = linear(gfeat.view(B * H, D), P['clusterFeatureAffine.weight'], B * H, x_planes=gfeat_pl)
    return gfeat, Kp, cmask, cidx.contiguous(), Wg.view(B, H, D)


@torch.no_grad()
def sue_tile_scores(meta, side, cand, *params):
    """click scores [B, T] of the candidates cand [B, T, D] for the users of ``side`` (from ``sue_user_side``): the
    candidate tail of SUEFunction.forward and the dot product (model.py:127)"""
    T = cand.shape[1]
    cand = cand.contiguous()
    if not meta['hca']:
        return RowDot.apply(side[0].unsqueeze(1).repeat(1, T, 1), cand)
    return RowDot.apply(_sue_tile_user(_Mod(), meta, side, cand, params), cand)


def _sue_tile_user(ctx, meta, side, cand, params):
    """the candidate tail of SUEFunction.forward with the cluster attention: user vectors [B, T, D] of the contiguous
    candidates cand [B, T, D]; the forward's tensors are left in ctx.sv"""
    P = dict(zip(sue_names(meta), params))
    B, T, D = cand.shape
    gfeat, Kp, cmask, cidx = side
    gcn = meta.get('gcn', True)
    L = meta['gcn_layers'] if gcn else 0
    C = P['proxy_node_embedding'].shape[0] if gcn else meta['category_num']
    H = gfeat.shape[1]
    return SUEFunction._clusters_tail(ctx, P, gfeat, cand, cmask, cidx, [0] * (L + 2), (B, H, D, T, C, H + C, C + 1), L, 0.0,
                                      keys=(None, Kp))


@torch.no_grad()
def sue_tile_explain(meta, side, cand, *params):
    """``sue_tile_scores`` and the explanation of each score: (scores [B, T], alpha [B, T, H], beta [B, T, C1],
    beta * (f . cand) [B, T, C1]) -- the model's own intra-cluster weights (cluster_intra_fwd), inter-cluster weights
    (attn_pool mode 1) and per-cluster score terms, whose sum over the clusters is the score up to fp32 rounding.  The
    scores are sue_tile_scores' bit for bit (the same kernels on the same shapes).  SUE_wo_HCA: (scores, the pooled
    attention's weights over the history expanded over the T candidates, None, None)."""
    B, T, D = cand.shape
    cand = cand.contiguous()
    if not meta['hca']:
        return sue_tile_scores(meta, side, cand, *params), side[1].unsqueeze(1).expand(-1, T, -1).contiguous(), None, None
    ctx = _Mod()
    user = _sue_tile_user(ctx, meta, side, cand, params)
    scores = RowDot.apply(user, cand)
    alpha, f, alpha2 = ctx.sv[2], ctx.sv[5], ctx.sv[9]
    C1 = side[2].shape[1]
    dots = _empty((B * T * C1,), cand.device)                                    # f_c . cand
    ops.rowdot_fwd(f, cand.view(B * T, 1, D).expand(-1, C1, -1).contiguous(), B * T * C1, D, dots)
    return scores, alpha.view(B, T, -1), alpha2.view(B, T, C1), (alpha2 * dots).view(B, T, C1)


@torch.no_grad()
def sue_tile_scores_factored(meta, side, cand_rows, *params):
    """click scores [B, T] of the candidates cand_rows [T, D], shared by the users of ``side`` (from
    ``sue_user_side(..., factored=True)``), through the factored cluster tail (nnr_cluster_tail_scores): the cluster affine
    is applied to the users' history rows (Wg) instead of to every (user, candidate) cluster feature.  The scores are those
    of SUEFunction.forward + RowDot in real arithmetic, not bit for bit; the candidate projections run once per row, not
    once per (user, row).  SUE_wo_HCA, whose user vector does not depend on the candidate: ``sue_tile_scores``."""
    T, D = cand_rows.shape
    if not meta['hca']:
        return sue_tile_scores(meta, side, cand_rows.unsqueeze(0).expand(side[0].shape[0], -1, -1), *params)
    P = dict(zip(sue_names(meta), params))
    gfeat, Kp, cmask, cidx, Wg = side
    B, H, _ = gfeat.shape
    C1 = cmask.shape[1]
    Au = P['intraCluster_K.weight'].shape[0]
    _, Qp, _, _, qk2 = SUEFunction._cand_side(P, cand_rows.contiguous(), 1, T, D)
    scores = _empty((B, T), gfeat.device)
    ops.cluster_tail_scores(Kp, gfeat, Wg, cidx, cmask.contiguous().view(torch.uint8), Qp, qk2, cand_rows.contiguous(),
                            P['clusterFeatureAffine.bias'], B, H, Au, D, C1, T, 1.0 / math.sqrt(float(Au)), scores)
    return scores


@torch.no_grad()
def sue_packed_scores_factored(meta, side, cand_rows, row_off, out, *params):
    """click scores of per-user candidate lists through the factored cluster tail (nnr_cluster_tail_scores_packed): user
    b of ``side`` (from ``sue_user_side(..., factored=True)``) has the candidates cand_rows [row_off[b], row_off[b + 1])
    (cand_rows [R, D] with R >= row_off[B], row_off [B + 1] int32 on the device); the score of its j-th candidate goes to
    out[b, j], and entries past its count are left as they are.  The candidate projections cost row_off[B] rows, not R.
    The scores are those of ``sue_tile_scores_factored`` on the same rows, bit for bit.  SUE_wo_HCA, whose user vector
    does not depend on the candidate: RowDot of the pooled user vector and each row, bit for bit the exact path's."""
    return _sue_packed_factored(meta, side, cand_rows, row_off, out, None, params)[0]


@torch.no_grad()
def sue_packed_explain_factored(meta, side, cand_rows, row_off, out, alpha, beta, contrib, *params):
    """``sue_packed_scores_factored`` that also explains each score it writes (nnr_cluster_tail_explain_packed): for user
    b's j-th candidate, alpha[b, j] [H] the intra-cluster weights of the history slots, beta[b, j] [C1] the inter-cluster
    weights and contrib[b, j] [C1] = beta * (f . cand) (alpha [B, n_max, H], beta / contrib [B, n_max, C1], contiguous,
    out contiguous).  Entries past a user's count are left as they are.  The scores equal sue_packed_scores_factored's
    bit for bit.  SUE_wo_HCA: alpha gets the pooled attention's weights over the history, beta and contrib are not
    used.  Returns (out, alpha, beta, contrib)."""
    return _sue_packed_factored(meta, side, cand_rows, row_off, out, (alpha, beta, contrib), params)


def _sue_packed_factored(meta, side, cand_rows, row_off, out, ex, params):
    """sue_packed_scores_factored (ex None) / sue_packed_explain_factored (ex = (alpha, beta, contrib))"""
    R, D = cand_rows.shape
    B, n_max = out.shape
    cand_rows = cand_rows.contiguous()
    total = row_off[B:]                                                      # int32 device scalar: the valid rows
    if not meta['hca']:
        user_of_row = torch.searchsorted(row_off[1:], torch.arange(R, dtype=torch.int32, device=out.device), right=True)
        dots = _empty((R,), out.device)
        ops.rowdot_fwd(side[0][user_of_row.clamp_(max=B - 1)].contiguous(), cand_rows, R, D, dots)
        j = torch.arange(n_max, device=out.device)
        lo = row_off[:B].long()
        valid = j[None, :] < (row_off[1:B + 1].long() - lo)[:, None]
        out.copy_(torch.where(valid, dots[(lo[:, None] + j[None, :]).clamp_(0, max(R - 1, 0))], out))
        if ex is not None:
            ex[0].copy_(torch.where(valid[:, :, None], side[1][:, None, :], ex[0]))
        return (out,) + (ex or ())
    P = dict(zip(sue_names(meta), params))
    gfeat, Kp, cmask, cidx, Wg = side
    H = gfeat.shape[1]
    C1 = cmask.shape[1]
    Au = P['intraCluster_K.weight'].shape[0]
    _, Qp, _, _, qk2 = SUEFunction._cand_side(P, cand_rows, 1, R, D, m_dev=total)
    args = (Kp, gfeat, Wg, cidx, cmask.contiguous().view(torch.uint8), row_off, Qp, qk2, cand_rows,
            P['clusterFeatureAffine.bias'], B, H, Au, D, C1, n_max, 1.0 / math.sqrt(float(Au)), out)
    if ex is None:
        ops.cluster_tail_scores_packed(*args)
        return (out,)
    ops.cluster_tail_explain_packed(*args, *ex)
    return (out,) + ex
