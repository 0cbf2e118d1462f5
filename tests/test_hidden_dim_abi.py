"""CPU test: the recurrence entry points reject hidden sizes outside the tensor-core kernels' range before any CUDA call.

Only unsupported sizes are passed here: a supported one would launch a kernel on the dummy pointers."""
import pytest

NNR_ERR_UNSUPPORTED = -4                                  # nnr_b200/csrc/common.cuh


@pytest.mark.parametrize('H', [150, 256])
def test_lstm_rejects_unsupported_hidden_dim_without_a_gpu(H):
    from nnr_b200 import _lib
    L = _lib.lib
    p = 256                                               # dummy, 16 B aligned, never dereferenced
    rc = L.nnr_lstm_fwd(p, p, p, p, p, 4, 8, H, p, p, p, p, None)
    assert rc == NNR_ERR_UNSUPPORTED
    msg = L.nnr_last_error().decode()
    assert 'nnr_lstm_fwd' in msg and 'hidden_dim %d' % H in msg and 'H % 4 == 0 and H <= 200' in msg
    rc = L.nnr_lstm_bwd(p, p, p, p, p, p, 4, 8, H, p, p, p, None)
    assert rc == NNR_ERR_UNSUPPORTED
    msg = L.nnr_last_error().decode()
    assert 'nnr_lstm_bwd' in msg and 'hidden_dim %d' % H in msg and 'H % 4 == 0 and H <= 200' in msg
