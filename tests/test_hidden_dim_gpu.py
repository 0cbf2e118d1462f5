"""hidden_dim other than 200: the tensor-core recurrence at every cluster size (2..5 CTAs of 40 units, ghost units up to the
cluster's padded width), and the drop-in Model at such sizes, against the fp64 / fp32 CPU oracle.

The op-level bounds are those of tests/test_ops_gpu.py::test_lstm_forward_backward, the model-level ones those of
tests/test_model_gpu.py."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import nnr_oracle as O
from tests.test_model_gpu import TOL, _args, _build, _check_grads, _oracle_grads
from tests.test_ops_gpu import _lstm_setup, _packed
from tests.util import GOLDEN_CASES, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RULE = r'H % 4 == 0 and H <= 200'


def _lstm_case(cuda, N, L, Hd, full, seed, guard=0):
    """inputs of one bidirectional recurrence; the device buffers are exact-size views of flat buffers followed by `guard`
    NaN-filled elements (the kernels must not touch them)"""
    from nnr_b200 import ops
    E = 24
    g = torch.Generator().manual_seed(seed)
    lens, x, w = _lstm_setup(N, L, Hd, E, g, full)
    ntok = int(lens.sum())
    len_ = lens.to(torch.int32).to(cuda)
    off = torch.cat([torch.zeros(1, dtype=torch.long), lens.cumsum(0)]).to(torch.int32).to(cuda)
    order = torch.sort(lens, descending=True, stable=True)[1].to(torch.int32).to(cuda)
    w_ih = torch.cat([w['weight_ih_l0'], w['weight_ih_l0_reverse']], 0)
    b = torch.cat([w['bias_ih_l0'] + w['bias_hh_l0'], w['bias_ih_l0_reverse'] + w['bias_hh_l0_reverse']], 0)
    xp = _packed(x, lens)
    w_hh = torch.stack([w['weight_hh_l0'], w['weight_hh_l0_reverse']], 0).to(cuda).contiguous()
    dh = torch.randn(N, L, 2 * Hd, generator=g)
    dcn = torch.randn(N, 2 * Hd, generator=g)

    def buf(rows, cols, fill=0.0):
        flat = torch.full((rows * cols + guard,), float('nan'), device=cuda)
        v = flat[:rows * cols].view(rows, cols)
        v.fill_(fill)
        return flat, v
    bufs = {k: buf(r, c) for k, (r, c) in dict(gx=(ntok, 8 * Hd), h=(ntok, 2 * Hd), cst=(ntok, 2 * Hd), cn=(N, 2 * Hd),
                                               dh=(ntok, 2 * Hd), dcn=(N, 2 * Hd)).items()}
    bufs['gx'][1].copy_((xp @ w_ih.t() + b).to(cuda))
    bufs['dh'][1].copy_(_packed(dh, lens).to(cuda))
    bufs['dcn'][1].copy_(dcn.to(cuda))

    def run():
        v = {k: t[1] for k, t in bufs.items()}
        ops.lstm_fwd(v['gx'], w_hh, len_, off, order, N, L, Hd, v['h'], v['cst'], v['cn'])
        torch.cuda.synchronize()
        fwd = (v['h'].clone(), v['cst'].clone(), v['cn'].clone())
        ops.lstm_bwd(v['gx'], v['cst'], w_hh, len_, off, order, N, L, Hd, v['dh'], v['dcn'])
        torch.cuda.synchronize()
        return fwd + (v['gx'].clone(),)
    return dict(lens=lens, x=x, w=w, xp=xp, w_ih=w_ih, dh=dh, dcn=dcn, ntok=ntok, bufs=bufs, run=run, tensors=(len_, off))


# every cluster size: CL = 2 (8, 40, 64), 3 (100, 120), 4 (128, 160), 5 (184, 196); ghost-free at 40, 120, 160
@pytest.mark.parametrize('Hd', [8, 40, 64, 100, 120, 128, 160, 184, 196])
@pytest.mark.parametrize('N,L,full', [(70, 12, False), (129, 33, False), (5, 128, False)])
def test_lstm_forward_backward_hidden_dim(cuda, Hd, N, L, full):
    _lstm_parity(cuda, Hd, N, L, full)


@pytest.mark.parametrize('Hd', [100, 128])
def test_lstm_forward_backward_hidden_dim_config2_history_shape(cuda, Hd):
    _lstm_parity(cuda, Hd, 3520, 128, 'mind')


def _lstm_parity(cuda, Hd, N, L, full):
    from nnr_b200 import ops
    c = _lstm_case(cuda, N, L, Hd, full, seed=7 + N + Hd)
    lens, x, ntok = c['lens'], c['x'], c['ntok']
    x64 = x.double().requires_grad_(True)
    w64 = {k: v.double().requires_grad_(True) for k, v in c['w'].items()}
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    h_ref, m_ref = O.bilstm(w64, '', x64, lens, impl='aten' if N > 1000 else 'loop')
    valid = (torch.arange(L)[None, :] < lens[:, None])
    ((h_ref * (c['dh'].double() * valid[..., None])).sum() + (m_ref * c['dcn'].double()).sum()).backward()
    h, _, cn, dgx = c['run']()
    e_h = (h.cpu().double() - _packed(h_ref.detach(), lens)).abs().max().item()
    e_c = (cn.cpu().double() - m_ref.detach()).abs().max().item()
    assert e_h < 5e-6 and e_c < 2e-5, (e_h, e_c)
    dgx = dgx.cpu().double()
    xp = c['xp'].double()
    dW_ref = torch.cat([w64['weight_ih_l0'].grad, w64['weight_ih_l0_reverse'].grad], 0)
    assert (dgx.t() @ xp - dW_ref).abs().max().item() / dW_ref.abs().max().item() < 2e-5
    db_ref = torch.cat([w64['bias_ih_l0'].grad, w64['bias_ih_l0_reverse'].grad], 0)
    assert (dgx.sum(0) - db_ref).abs().max().item() / db_ref.abs().max().item() < 2e-5
    dx_ref = _packed(x64.grad, lens)
    assert (dgx @ c['w_ih'].double() - dx_ref).abs().max().item() / dx_ref.abs().max().item() < 2e-5
    len_, off = c['tensors']
    tok_row = torch.repeat_interleave(torch.arange(N), lens).to(torch.int32).to(cuda)
    hprev = torch.empty(ntok, 2 * Hd, device=cuda)
    ops.lstm_shift_h(h, len_, off, tok_row, N, L, Hd, hprev)
    hp = hprev.cpu().double()
    for d, sfx in enumerate(('', '_reverse')):
        dWhh = dgx[:, d * 4 * Hd:(d + 1) * 4 * Hd].t() @ hp[:, d * Hd:(d + 1) * Hd]
        ref = w64['weight_hh_l0' + sfx].grad
        assert (dWhh - ref).abs().max().item() / ref.abs().max().item() < 2e-5, sfx


@pytest.mark.parametrize('Hd', [100, 184])
def test_lstm_writes_nothing_outside_its_tensors(cuda, Hd):
    """h, c_stash, c_n and gx (stash, then dL/dgx) are exact-size views (rows = tokens) followed by NaN guards: ghost units
    never reach global memory, and neither do the reads (a NaN read would poison the results)"""
    c = _lstm_case(cuda, 129, 33, Hd, False, seed=11, guard=4096)
    out = c['run']()
    for k, (flat, v) in c['bufs'].items():
        assert torch.isnan(flat[v.numel():]).all(), k
    for t in out:
        assert torch.isfinite(t).all()


def test_lstm_hidden_dim_is_deterministic(cuda):
    runs = [_lstm_case(cuda, 129, 33, 100, False, seed=5)['run']() for _ in range(2)]
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def _model_case(name, Hd, **over):
    from nnr_b200.synthetic import SyntheticMIND
    kw = dict(GOLDEN_CASES[name], **over)
    cfg = O.make_config(hidden_dim=Hd, dropout_rate=0.0, **kw)
    syn = SyntheticMIND(news_num=300 if name == 'dev_shape' else 200, vocabulary_size=cfg.vocabulary_size,
                        subCategory_num=cfg.subCategory_num, max_title_length=cfg.max_title_length,
                        max_abstract_length=cfg.max_abstract_length, max_history_num=cfg.max_history_num, lengths='uniform', seed=3)
    return cfg, syn.batch(3, seed=1)


def _model_parity(cuda, cfg, batch, label):
    from nnr_b200.trainer import negative_log_softmax
    p = O.formula_params(cfg)
    ref_logits, _, _ = O.forward_backward(p, cfg, batch, sort_fn=O.stable_sort)
    m = _build(cfg, p, cuda)
    with torch.no_grad():
        out = m(*_args(batch, cuda))
    assert rel_err(out, ref_logits) < TOL, label
    _, g64, loss64, tol = _oracle_grads(cfg, batch, p)
    m = _build(cfg, p, cuda, train=True)
    loss = negative_log_softmax(m(*_args(batch, cuda)))
    loss.backward()
    assert abs(loss.item() - loss64.item()) < 1e-4 * max(1.0, abs(loss64.item())), label
    _check_grads(label, m, g64, tol)


# 100: h_{t-1} of the weight gradient as fp32 instead of 16-bit planes (the reverse half would start at an unaligned column)
@pytest.mark.parametrize('Hd', [64, 100, 128, 184])
@pytest.mark.parametrize('name', ['tiny', 'dev_shape'])
def test_model_matches_oracle_at_hidden_dim(cuda, name, Hd):
    cfg, batch = _model_case(name, Hd)
    _model_parity(cuda, cfg, batch, '%s/H=%d' % (name, Hd))


@pytest.mark.parametrize('encoders', [('CNE_wo_CA', 'SUE_wo_HCA'), ('CNE_Title', 'SUE')])
def test_model_variants_match_oracle_at_hidden_dim_128(cuda, encoders):
    cfg, batch = _model_case('tiny', 128, news_encoder=encoders[0], user_encoder=encoders[1])
    _model_parity(cuda, cfg, batch, '%s+%s/H=128' % encoders)


def test_cuda_graph_step_equals_eager_step_at_hidden_dim_128(cuda):
    from nnr_b200.synthetic import SyntheticMIND, batch_args
    from nnr_b200.trainer import TrainStep
    cfg = O.make_config(hidden_dim=128, vocabulary_size=800, max_history_num=10, max_title_length=16, max_abstract_length=40,
                        subCategory_num=40, gcn_layer_num=2, dropout_rate=0.0)
    syn = SyntheticMIND(news_num=300, vocabulary_size=800, subCategory_num=40, max_title_length=16, max_abstract_length=40,
                        max_history_num=10, lengths='mind', seed=7)
    batches = [batch_args(syn.batch(6, seed=s), cuda) for s in (1, 2, 3)]
    p = O.formula_params(cfg)
    steps = []
    for graph in (False, True):
        m = _build(cfg, p, cuda, train=True)
        steps.append((m, TrainStep(m, lr=1e-3, gradient_clip_norm=4.0, world_size=1, cuda_graph=graph)))
    (m_e, ts_e), (m_g, ts_g) = steps
    for i in range(4):
        b = batches[i % 3]
        le = ts_e.step(*[x.clone() if torch.is_tensor(x) else x for x in b]).item()
        lg = ts_g.step(*[x.clone() if torch.is_tensor(x) else x for x in b]).item()
        assert abs(le - lg) <= 1e-6 * max(1.0, abs(le)), (i, le, lg)
    assert len(ts_g._graphs) == 1
    for (k, a), (_, b) in zip(m_e.named_parameters(), m_g.named_parameters()):
        assert (a - b).abs().max().item() <= 1e-6 * max(1.0, a.abs().max().item()), k


def _bf16_check_hidden_dim_128(cuda):
    """the model-level tolerance of tests/test_model_gpu.py::_bf16_variant_check, against the fp64 oracle"""
    from nnr_b200 import ops
    from nnr_b200.trainer import negative_log_softmax
    assert ops.default_algo() == ops.ALGO_BF16
    cfg, batch = _model_case('dev_shape', 128)
    p = O.formula_params(cfg)
    g32, g64, loss64, _ = _oracle_grads(cfg, batch, p)
    logits64, _, _ = O.forward_backward(p, cfg, batch, dtype=torch.float64, sort_fn=O.stable_sort)
    m = _build(cfg, p, cuda, train=True)
    logits = m(*_args(batch, cuda))
    loss = negative_log_softmax(logits)
    loss.backward()
    e_logits = rel_err(logits, logits64)
    e_loss = abs(loss.item() - loss64.item())
    assert e_logits <= 2e-2 and e_loss <= 1e-2, (e_logits, e_loss)
    named = dict(m.named_parameters())
    gmax = max(float(v.abs().max()) for v in g64.values())
    worst = []
    for k in [k for k in named if not k.startswith('user_encoder.news_encoder.')]:
        a, b = named[k].grad.detach().cpu().double().flatten(), g64[k].flatten()
        noise = (g32[k].double().flatten() - b).abs().max().item()
        err = (a - b).abs().max().item()
        # + 1e-7 max|g64| over the model, as in _oracle_grads: a tensor whose true gradient is ~0 (intraCluster_K / Q when
        # every cluster is a singleton) is pure rounding noise
        worst.append((err / (5e-2 * b.abs().max().item() + 8 * noise + 1e-7 * gmax), k, err))
        if b.abs().max().item() > 100 * noise and b.norm() > 0:
            cos = float(a @ b / (a.norm() * b.norm() + 1e-300))
            assert cos >= 0.999, (k, cos)
    worst.sort(reverse=True)
    assert worst[0][0] < 1.0, worst[:5]


def _child(code, env_over, marker):
    env = dict(os.environ, **env_over)
    r = subprocess.run([sys.executable, '-c', code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and marker in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_bf16_variant_model_level_tolerance_at_hidden_dim_128_subprocess(cuda):
    _child("import torch, tests.test_hidden_dim_gpu as t; t._bf16_check_hidden_dim_128(torch.device('cuda:0')); print('bf16-ok')",
           dict(NNR_GEMM_ALGO='bf16'), 'bf16-ok')


@pytest.mark.parametrize('Hd', [150, 204, 256])
def test_unsupported_hidden_dim_is_rejected(cuda, Hd):
    with pytest.raises(RuntimeError, match=RULE):
        _lstm_case(cuda, 5, 8, Hd, False, seed=1)['run']()
    cfg, batch = _model_case('tiny', Hd)
    m = _build(cfg, O.formula_params(cfg), cuda)
    with pytest.raises(RuntimeError, match=RULE):
        with torch.no_grad():
            m(*_args(batch, cuda))


def test_ffma_recurrence_names_its_switch_at_hidden_dim_128_subprocess(cuda):
    code = ("import torch, pytest, tests.test_hidden_dim_gpu as t\n"
            "with pytest.raises(RuntimeError, match='NNR_LSTM_ALGO=ffma'):\n"
            "    t._lstm_case(torch.device('cuda:0'), 5, 8, 128, False, seed=1)['run']()\n"
            "print('ffma-rejects')")
    _child(code, dict(NNR_LSTM_ALGO='ffma'), 'ffma-rejects')
