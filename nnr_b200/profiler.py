"""CUDA-event breakdown of a training step by C-ABI op, and the roofline entry bench.py prints.

``capture()`` wraps every function of ``nnr_b200.ops`` that launches kernels with a pair of CUDA
events recorded on the launching (current) stream; nothing synchronises until ``summary()``.
Algorithmic work per call (SURVEY.md 8d / DESIGN.md "algorithmic work"):
  gemm        2*M*N*K flop, M (or K) replaced by the device-side valid-token count when given
  lstm_fwd    2 * (4H*H) flop per token per direction  (recurrent product only)
  lstm_bwd    2 * (4H*H) flop per token per direction  (dh_{t-1} product; dW_hh is a separate GEMM)
  embed_gather_fwd   tokens * (4 + 2*4*E) bytes      embed_gather_bwd   tokens * (4 + 4*E) + V*E*4 bytes
  attn_pool_*        tokens * D * 4 * (reads+writes) bytes
"""
import contextlib
import ctypes
import json
import os

import torch

from . import _lib, ops

_KERNEL_TAGS = ['gemm_tc_kernel', 'tc_split_kernel', 'tc_splitk_reduce_kernel', 'gemm_simt_kernel']


def _tc_class(M, N, K, transA, transB, m_dev, k_dev):
    """mirror of nnr_gemm_tc_supported (gemm_tc.cu): which nnr_gemm calls run on the tcgen05 kernel"""
    if os.environ.get('NNR_GEMM_ALGO') == 'simt':
        return False
    if float(M) * N * K < 2.0e6 or K < 8:
        return False
    if m_dev is not None and transA:
        return False
    if k_dev is not None and not (transA and not transB):
        return False
    return True

_TIMED = ['seq_prepare', 'embed_gather_fwd', 'embed_gather_planes_fwd', 'embed_gather_bwd', 'gemm', 'colsum', 'segment_colsum', 'lstm_fwd', 'lstm_fwd_planes',
          'lstm_bwd', 'lstm_bwd_planes', 'lstm_shift_h', 'lstm_shift_h_planes', 'gate_bwd_pre', 'gate_bwd_planes', 'attn_pool_fwd', 'attn_pool_bwd', 'news_fuse_fwd', 'news_fuse_bwd', 'news_fuse_split_bwd', 'news_fuse_tables_bwd',
          'graph_to_csr', 'gcn_aggregate', 'cluster_intra_fwd', 'cluster_intra_bwd', 'rowdot_fwd', 'rowdot_bwd',
          'dropout', 'flat_clip_adam', 'sue_graph_build', 'relu_bwd_split_colsum']


def _dev_int(t):
    return int(t.item()) if t is not None else None


class Capture:
    def __init__(self):
        self.records = []
        self.t0 = self.t1 = None

    def _work(self, name, args, kw):
        """returns a closure evaluated after synchronisation -> (flops, bytes)"""
        if name == 'gemm':
            A, B, C, M, N, K = args[:6]
            m_dev, k_dev = kw.get('m_dev'), kw.get('k_dev')
            tc = _tc_class(M, N, K, args[9], args[10], m_dev, k_dev)
            return lambda: (2.0 * (min(M, _dev_int(m_dev)) if m_dev is not None else M) * N *
                            (min(K, _dev_int(k_dev)) if k_dev is not None else K), None, tc)
        if name in ('lstm_fwd', 'lstm_fwd_planes', 'lstm_bwd', 'lstm_bwd_planes'):
            if name in ('lstm_fwd', 'lstm_fwd_planes'):
                off, N, H = args[3], args[5], args[7]
            else:
                off, N, H = args[4], args[6], args[8]
            return lambda: (2.0 * 4 * H * H * 2 * int(off[N].item()), None)
        if name in ('embed_gather_fwd', 'embed_gather_planes_fwd'):      # planes: hi + lo bf16 = the same 4 bytes per element
            table, ids, len_, off = args[:4]
            E = table.shape[1]
            return lambda: (None, float(off[ids.shape[0]].item()) * (4 + 8 * E))
        if name == 'embed_gather_bwd':
            dout, ids, len_, off, dtable = args[:5]
            V, E = dtable.shape
            return lambda: (None, float(off[ids.shape[0]].item()) * (4 + 4 * E) + V * E * 4.0)
        if name in ('attn_pool_fwd', 'attn_pool_bwd'):
            S, D, A = kw['S'], kw['D'], kw.get('A', 0) or 0
            seg_off, fixed = kw.get('seg_off'), kw.get('fixed_len', 0)
            mode0 = kw.get('mode') == 0
            fwd = name == 'attn_pool_fwd'
            acc = bool(kw.get('accumulate_dx', False))

            def pool_bytes():
                rows = float(seg_off[S].item()) if seg_off is not None else float(S * fixed)
                per_row = D * 4 + (A * 4 if mode0 else 0) + 4                  # X once (+ U), alpha
                if not fwd:
                    per_row += D * 4 * (2 if acc else 1) + (A * 4 if mode0 else 0)   # dX (read-modify-write if accumulating), dU
                return (None, rows * per_row + S * D * 4.0)
            return pool_bytes
        if name == 'colsum':
            X, ldx, M, N = args[:4]
            m_dev = kw.get('m_dev', args[6] if len(args) > 6 else None)
            return lambda: (None, (min(M, _dev_int(m_dev)) if m_dev is not None else M) * N * 4.0)
        if name == 'flat_clip_adam':
            n = args[0].numel()
            return lambda: (None, n * 28.0)                                       # read p, g (x2: norm + update), m, v; write p, m, v
        if name == 'gcn_aggregate':
            B, Gn, D = args[4], args[5], args[6]
            return lambda: (None, 2.0 * B * Gn * D * 4)                           # features in once, aggregated features out
        return lambda: (None, None)

    def wrap(self, name, fn):
        def wrapped(*args, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            work = self._work(name, args, kw)
            e0.record()
            r = fn(*args, **kw)
            e1.record()
            label = name
            if name == 'gemm':
                label = 'gemm[%dx%dx%d %s%s e%d]' % (args[3], args[4], args[5], 'T' if args[9] else 'N', 'T' if args[10] else 'N',
                                                   kw.get('epilogue', args[11] if len(args) > 11 else 0))
            alias = {'embed_gather_planes_fwd': 'embed_gather_fwd', 'lstm_bwd_planes': 'lstm_bwd', 'lstm_fwd_planes': 'lstm_fwd', 'lstm_shift_h_planes': 'lstm_shift_h',
                     'gate_bwd_planes': 'gate_bwd_pre'}   # same op, planes output
            self.records.append((alias.get(name, name), e0, e1, work, label))
            return r
        return wrapped

    def summary(self, steps=1):
        torch.cuda.synchronize()
        agg = {}
        self.detail = {}
        tc_flops = simt_flops = 0.0
        for name, e0, e1, work, label in self.records:
            ms = e0.elapsed_time(e1)
            w = work()
            fl, by = w[0], w[1]
            if name == 'gemm':
                if w[2]:
                    tc_flops += fl
                else:
                    simt_flops += fl
            for key, table in ((name, agg), (label, self.detail)):
                a = table.setdefault(key, {'ms': 0.0, 'calls': 0, 'flops': 0.0, 'bytes': 0.0})
                a['ms'] += ms
                a['calls'] += 1
                a['flops'] += fl or 0.0
                a['bytes'] += by or 0.0
        self.detail = {k: {'ms': round(a['ms'] / steps, 3), 'calls': a['calls'] / steps,
                           'tflops': round(a['flops'] / max(a['ms'], 1e-9) / 1e9, 1)}
                       for k, a in sorted(self.detail.items(), key=lambda kv: -kv[1]['ms']) if k.startswith('gemm[')}
        # kernel-level times of the composite gemm op (events recorded inside the library around each kernel)
        buf = (ctypes.c_double * (3 * len(_KERNEL_TAGS)))()
        _lib.lib.nnr_profile_read(buf, len(_KERNEL_TAGS))
        if 'gemm' in agg:
            agg['gemm (op total: split + main + reduce)'] = agg.pop('gemm')
            agg['gemm (op total: split + main + reduce)']['flops'] = 0.0
        for i, tag in enumerate(_KERNEL_TAGS):
            if buf[3 * i + 1] > 0:
                agg[tag] = {'ms': buf[3 * i], 'calls': buf[3 * i + 1], 'bytes': 0.0,
                            'flops': tc_flops if tag == 'gemm_tc_kernel' else (simt_flops if tag == 'gemm_simt_kernel' else 0.0)}
        out = {}
        for k, a in sorted(agg.items(), key=lambda kv: -kv[1]['ms'] if not kv[0].startswith('gemm (op') else 1.0):
            out[k] = {'ms': a['ms'] / steps, 'calls': a['calls'] / steps}
            if a['flops']:
                out[k]['tflops'] = a['flops'] / (a['ms'] * 1e-3) / 1e12
            if a['bytes']:
                out[k]['gbs'] = a['bytes'] / (a['ms'] * 1e-3) / 1e9
        return out


@contextlib.contextmanager
def capture():
    from . import engine
    cap = Capture()
    _lib.lib.nnr_profile_enable(1)
    saved = {}
    lanes_were = engine.concurrent
    engine.concurrent = False          # per-op events time one op at a time: no second lane (engine.Lanes) underneath them
    for name in _TIMED:
        saved[name] = getattr(ops, name)
        setattr(ops, name, cap.wrap(name, saved[name]))
    try:
        yield cap
    finally:
        _lib.lib.nnr_profile_enable(0)
        engine.concurrent = lanes_were
        for name, fn in saved.items():
            setattr(ops, name, fn)


def measured_peaks(root):
    path = os.path.join(root, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p.get('bf16_tflops_sustained', p['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1400.0, 'source': 'fallback'}


def _ncu_traffic(root, kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json), or None"""
    path = os.path.join(root, 'profiles', 'traffic.json')
    if not os.path.isfile(path):
        return None
    with open(path) as f:
        entry = json.load(f).get(kernel)
    return entry['dram_bytes_per_launch'] if entry else None


def _ncu_traffic_source(root, kernel):
    path = os.path.join(root, 'profiles', 'traffic.json')
    if not os.path.isfile(path):
        return None
    with open(path) as f:
        entry = json.load(f).get(kernel)
    return ('static: ' + entry['source']) if entry else None


def roofline(breakdown, tokens_per_step, batch, root):
    """roofline entry for the dominant op of the step (largest share of device time)"""
    if not breakdown:
        return None
    name, top = next(iter(breakdown.items()))
    peaks = measured_peaks(root)
    traffic = _ncu_traffic(root, name)
    total = sum(v['ms'] for k, v in breakdown.items() if k not in _KERNEL_TAGS)
    if 'tflops' in top:
        # algorithmic flops (the 3 split products count once).  Denominator: the tensor rate of the MMA kind the
        # kernel issues -- bf16 cuBLAS (measured, sustained) for bf16x3 / bf16, half of it for tf32x3.
        algo = ops.default_algo()
        tf32 = (algo == ops.ALGO_TF32X3) and name == 'gemm_tc_kernel'
        peak = peaks['bf16_tflops'] / (2.0 if tf32 else 1.0)
        note = '%s bf16 cuBLAS %s TFLOP/s sustained%s; algorithmic flops, split products not counted' % (
            peaks['source'], peaks['bf16_tflops'], ' x 0.5 (kind::tf32)' if tf32 else '')
        products = 3 if algo in (ops.ALGO_TF32X3, ops.ALGO_BF16X3) and name == 'gemm_tc_kernel' else 1
        return {'kernel': name, 'bound': 'tensor', 'achieved': top['tflops'], 'peak': peak, 'unit': 'TFLOP/s',
                'frac': top['tflops'] / peak, 'traffic': traffic, 'traffic_source': _ncu_traffic_source(root, name),
                'share_of_step': top['ms'] / total,
                'gemm_algo': {1: 'simt', 2: 'tf32x3', 3: 'bf16', 4: 'bf16x3'}.get(algo, str(algo)), 'peak_note': note,
                # fp32-grade results on 16-bit tensor cores cost `products` MMAs per algorithmic flop: the fraction of
                # the tensor pipe's measured peak that the kernel actually sustains is products x frac
                'mma_per_algorithmic_flop': products, 'frac_of_peak_in_issued_mma': products * top['tflops'] / peak}
    if 'gbs' in top:
        return {'kernel': name, 'bound': 'hbm', 'achieved': top['gbs'], 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                'frac': top['gbs'] / peaks['hbm_gbs'], 'traffic': traffic, 'traffic_source': _ncu_traffic_source(root, name),
                'share_of_step': top['ms'] / total,
                'peak_note': '%s HBM copy bandwidth' % peaks['source']}
    return {'kernel': name, 'bound': 'hbm', 'achieved': None, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': None,
            'traffic': traffic, 'share_of_step': top['ms'] / total}


def roofline_table(breakdown, root):
    """one row per op that has algorithmic work attached: achieved rate against the measured peak that bounds it"""
    peaks = measured_peaks(root)
    algo = ops.default_algo()
    products = 3 if algo in (ops.ALGO_TF32X3, ops.ALGO_BF16X3) else 1
    rows = []
    for name, v in breakdown.items():
        if 'tflops' in v:
            tensor = name in ('gemm_tc_kernel', 'lstm_fwd', 'lstm_bwd')
            if not tensor:
                continue
            rows.append({'kernel': name, 'bound': 'tensor', 'ms': round(v['ms'], 3), 'achieved': round(v['tflops'], 1),
                         'unit': 'TFLOP/s (algorithmic)', 'peak': peaks['bf16_tflops'], 'frac': round(v['tflops'] / peaks['bf16_tflops'], 4),
                         'mma_per_algorithmic_flop': products,
                         'frac_of_peak_in_issued_mma': round(products * v['tflops'] / peaks['bf16_tflops'], 4)})
        elif 'gbs' in v:
            rows.append({'kernel': name, 'bound': 'hbm', 'ms': round(v['ms'], 3), 'achieved': round(v['gbs'], 1), 'unit': 'GB/s (algorithmic)',
                         'peak': peaks['hbm_gbs'], 'frac': round(v['gbs'] / peaks['hbm_gbs'], 4)})
    return rows
