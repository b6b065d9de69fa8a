"""Prediction without a GPU: the fp64 reference of the class probabilities, and the argument checks of
agcn_head_predict / agcn_stack_predict (they reject bad calls before anything touches the device)."""
import ctypes

import numpy as np
import pytest
import torch

from predict_oracle import head_predict

AGCN_ERR_INVALID = -1


def _head(B, Fh, Fm, Nt, seed):
    g = torch.Generator().manual_seed(seed)
    sizes = torch.randint(3, 30, (B,), generator=g).tolist()
    H = [torch.randn(n, Fh, generator=g, dtype=torch.float64) for n in sizes]
    p = {"dense_W": torch.randn(Fh, Fm, generator=g, dtype=torch.float64) * 0.05,
         "dense_b": torch.randn(Fm, generator=g, dtype=torch.float64) * 0.02,
         "head_W": torch.randn(Fm, Nt, generator=g, dtype=torch.float64),
         "head_b": torch.randn(Nt, generator=g, dtype=torch.float64) * 0.05}
    mol = np.tanh(np.stack([(h.numpy() @ p["dense_W"].numpy() + p["dense_b"].numpy()).sum(0) for h in H]))
    logits = mol @ p["head_W"].numpy() + p["head_b"].numpy()
    return H, p, logits


def _np_softmax(x):
    e = np.exp(x - x.max(-1, keepdims=True))
    return e / e.sum(-1, keepdims=True)


def test_oracle_multitask_probabilities_are_a_softmax_per_task():
    B, T = 9, 12
    H, p, logits = _head(B, 16, 32, 2 * T, seed=1)
    probs = head_predict(H, p, "sigmoid_ce")
    assert probs.shape == (B, T, 2) and probs.dtype == torch.float64
    assert np.allclose(probs.sum(-1).numpy(), 1.0, rtol=0, atol=1e-12)
    x = logits.reshape(B, T, 2)
    assert np.allclose(probs.numpy(), _np_softmax(x), rtol=0, atol=1e-12)
    # the two-logit softmax is the logistic function of the logit difference
    assert np.allclose(probs[..., 1].numpy(), 1.0 / (1.0 + np.exp(x[..., 0] - x[..., 1])), rtol=0, atol=1e-12)


def test_oracle_single_task_probabilities_are_a_softmax_per_sample():
    B, C = 7, 40
    H, p, logits = _head(B, 16, 32, C, seed=2)
    probs = head_predict(H, p, "softmax_ce")
    assert probs.shape == (B, C)
    assert np.allclose(probs.sum(-1).numpy(), 1.0, rtol=0, atol=1e-12)
    assert np.allclose(probs.numpy(), _np_softmax(logits), rtol=0, atol=1e-12)
    with pytest.raises(ValueError):
        head_predict(H, p, "hinge")


def _fake(n):
    """Distinct non-NULL addresses: the calls below must fail on their argument checks, before any is used."""
    return [ctypes.c_void_p(0x1000 * (i + 1)) for i in range(n)]


def _last_error():
    from agcn_b200 import _lib
    return _lib.lib().agcn_last_error().decode()


def test_head_predict_rejects_null_plan_and_mismatched_loss_pointers():
    from agcn_b200 import _lib
    lib = _lib.lib()
    H, dW, db, hW, hb, tg, w, probs, loss, work = _fake(10)
    stream = ctypes.c_void_p(0)

    def call(plan, tg, w, loss, loss_kind=0, Fm=64, Nt=24):
        return lib.agcn_head_predict(plan, H, dW, db, hW, hb, tg, w, 1.0, loss_kind, 64, Fm, Nt, probs, loss, work,
                                     1 << 20, stream)

    assert call(None, None, None, None) == AGCN_ERR_INVALID
    assert "head_predict" in _last_error() and "null pointer" in _last_error()
    assert call(None, tg, w, None) == AGCN_ERR_INVALID             # targets without a loss output
    assert "all NULL or all set" in _last_error()
    assert call(None, tg, None, loss) == AGCN_ERR_INVALID          # weights missing
    assert "all NULL or all set" in _last_error()
    assert call(None, None, None, loss) == AGCN_ERR_INVALID        # a loss output without targets
    assert "all NULL or all set" in _last_error()
    size = ctypes.c_size_t()
    assert lib.agcn_head_predict_workspace_bytes(None, 64, 64, 24, ctypes.byref(size)) == AGCN_ERR_INVALID
    assert "head_predict_workspace_bytes" in _last_error()


def test_stack_predict_rejects_null_plan_and_mismatched_loss_pointers():
    from agcn_b200 import _lib
    lib = _lib.lib()
    descs = (_lib.Desc * 2)(_lib.Desc(75, 64, 3, 0, 0, 0, 1, _lib.SAVE_FOR_BACKWARD),
                            _lib.Desc(64, 64, 3, 0, 0, 0, 1, _lib.SAVE_FOR_BACKWARD))
    offs = (ctypes.c_int64 * 14)(*range(14))
    stack = ctypes.c_void_p()
    _lib.check(lib.agcn_stack_create(descs, 2, 64, 24, _lib.LOSS["sigmoid_ce"], offs, ctypes.byref(stack)))
    try:
        X, L, tg, w, params, probs, loss, work = _fake(8)
        stream = ctypes.c_void_p(0)

        def call(plan, tg, w, loss):
            return lib.agcn_stack_predict(stack, plan, X, L, tg, w, 1.0, params, probs, loss, work, 1 << 20, stream)

        assert call(None, None, None, None) == AGCN_ERR_INVALID
        assert "stack_predict" in _last_error() and "null pointer" in _last_error()
        assert call(None, tg, w, None) == AGCN_ERR_INVALID
        assert "all NULL or all set" in _last_error()
        assert call(None, None, w, loss) == AGCN_ERR_INVALID
        assert "all NULL or all set" in _last_error()
        size = ctypes.c_size_t()
        assert lib.agcn_stack_predict_workspace_bytes(stack, None, ctypes.byref(size)) == AGCN_ERR_INVALID
        assert "stack_predict_workspace_bytes" in _last_error()
    finally:
        lib.agcn_stack_destroy(stack)


def test_functional_head_predict_needs_targets_and_weights_together():
    from agcn_b200.functional import head_predict as fhp
    with pytest.raises(ValueError):
        fhp(None, None, None, None, None, None, "sigmoid_ce", targets=torch.zeros(2, 4))
