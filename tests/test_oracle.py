"""CPU tests: the oracle restatement against the golden outputs of the real reference, and (where
/root/reference exists) against the live reference."""
import numpy as np
import pytest
import torch

from oracle import nnr_oracle as O
from oracle import reference_import as R
from tests.util import GOLDEN_CASES, grad_digest, load_big_golden, load_golden


@pytest.mark.parametrize('name', list(GOLDEN_CASES))
def test_oracle_matches_golden_logits(name):
    cfg, batch, z = load_golden(name)
    p = O.formula_params(cfg)
    with torch.no_grad():
        out_default = O.model_forward(p, cfg, batch)
        out_stable = O.model_forward(p, cfg, batch, sort_fn=O.stable_sort)
    np.testing.assert_allclose(out_default.numpy(), z['logits_default_sort'], rtol=0, atol=2e-5)
    np.testing.assert_allclose(out_stable.numpy(), z['logits_stable_sort'], rtol=0, atol=2e-5)


def test_oracle_matches_full_length_golden_logits():
    """full_b8 (8 impressions, every title 32 / abstract 128 tokens): inputs regenerated from the seeds and hash-checked"""
    cfg, batch, z = load_big_golden('full_b8')
    p = O.formula_params(cfg)
    with torch.no_grad():
        out = O.model_forward(p, cfg, batch, sort_fn=O.stable_sort, lstm_impl='aten')
    np.testing.assert_allclose(out.numpy(), z['logits_stable_sort'], rtol=0, atol=2e-5 * float(np.abs(z['logits_stable_sort']).max()))


@pytest.mark.parametrize('name', ['tiny', 'ablation', 'layer_norm', 'no_residual'])
def test_oracle_matches_golden_gradients(name):
    cfg, batch, z = load_golden(name)
    cfg.dropout_rate = 0.0
    p = O.formula_params(cfg)
    logits, loss, grads = O.forward_backward(p, cfg, batch, sort_fn=O.stable_sort)
    _, _, grads64 = O.forward_backward(p, cfg, batch, dtype=torch.float64, sort_fn=O.stable_sort)
    np.testing.assert_allclose(logits.numpy(), z['train_logits'], atol=2e-5)
    assert abs(float(loss) - float(z['train_loss'])) < 1e-5
    gscale = max(float(z['grad_' + k][2]) for k in grads)            # largest gradient entry overall
    for k, g in grads.items():
        ref = z['grad_' + k]
        mine = grad_digest(g)
        # fp32 rounding of the oracle where the test runs (its fp32 digest against its fp64 one): gradients that are sums with heavy
        # cancellation (the self-attention biases, ~1e-7 against a largest entry of ~0.07) move by that much with the CPU's
        # summation order (thread count, vector width), here and in the golden run alike -- as in test_model_gpu's tolerance
        noise = np.abs(mine - grad_digest(grads64[k]))
        tol = 1e-4 * max(ref[2], 1e-4 * gscale) + 8 * max(noise[2], noise[3:].max())
        assert abs(mine[2] - ref[2]) <= tol, k
        assert np.all(np.abs(mine[3:] - ref[3:]) <= tol), k
        assert abs(mine[0] - ref[0]) <= 1e-4 * max(ref[1], 1e-12) + 1e-9 + 8 * noise[0], k


def test_loop_lstm_equals_aten_lstm():
    cfg, batch, _ = load_golden('tiny')
    p = O.formula_params(cfg)
    with torch.no_grad():
        a = O.model_forward(p, cfg, batch, lstm_impl='loop')
        b = O.model_forward(p, cfg, batch, lstm_impl='aten')
    assert (a - b).abs().max().item() < 2e-6


def test_oracle_fp64_consistency():
    cfg, batch, _ = load_golden('tiny')
    cfg.dropout_rate = 0.0
    p = O.formula_params(cfg)
    l32, _, g32 = O.forward_backward(p, cfg, batch, sort_fn=O.stable_sort)
    l64, _, g64 = O.forward_backward(p, cfg, batch, dtype=torch.float64, sort_fn=O.stable_sort)
    assert (l32.double() - l64).abs().max().item() < 1e-5


@pytest.mark.skipif(not R.available(), reason='needs a checkout of the original NNR project at NNR_REFERENCE_ROOT; '
                    'test_oracle_matches_golden_logits checks against its stored outputs')
def test_oracle_matches_live_reference():
    cfg, batch, _ = load_golden('tiny')
    p = O.formula_params(cfg, salt=3)                                 # different weights than the golden run
    m = R.build_reference_model(cfg, p)
    m.eval()
    with torch.no_grad():
        ref = R.run_reference(m, batch)
        mine = O.model_forward(p, cfg, batch)
    assert (ref - mine).abs().max().item() < 2e-6


def test_scatter_restatement_properties():
    torch.manual_seed(0)
    src = torch.randn(2, 3, 11)
    idx = torch.randint(0, 4, (2, 3, 11))
    sm = O.scatter_softmax(src, idx, 2)
    sums = O.scatter_sum(sm, idx, 2, 5)
    present = O.scatter_sum(torch.ones_like(sm), idx, 2, 5) > 0
    assert torch.allclose(sums[present], torch.ones_like(sums[present]), atol=1e-6)
    assert torch.all(sums[~present] == 0)


def test_clip_adam_restatement_against_torch():
    torch.manual_seed(1)
    w = {'a': torch.randn(7, 5), 'b': torch.randn(11)}
    tw = {k: v.clone().requires_grad_(True) for k, v in w.items()}
    opt = torch.optim.Adam(tw.values(), lr=1e-2)
    state = {}
    for step in range(1, 4):
        g = {k: torch.randn_like(v) * 3 for k, v in w.items()}
        for k in tw:
            tw[k].grad = g[k].clone()
        torch.nn.utils.clip_grad_norm_(tw.values(), 4.0)
        opt.step()
        O.clip_and_adam(w, g, state, step, lr=1e-2)
        for k in w:
            assert torch.allclose(w[k], tw[k].detach(), atol=1e-6), (k, step)
