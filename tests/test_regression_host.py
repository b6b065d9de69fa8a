"""The regression head (loss="weighted_l2") without a GPU: the loss constant of the C ABI and its Python binding, the
argument checks of the head / stack calls for the new kind (they reject bad calls before anything touches the device),
SimpleAGCNStep's regressor surface, the synthetic regression labels, and the fp64 reference against its closed form."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import regression_oracle as RO

AGCN_ERR_INVALID = -1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _last_error():
    from agcn_b200 import _lib
    return _lib.lib().agcn_last_error().decode()


def _fake(n):
    """Distinct non-NULL addresses: the calls below must fail on their argument checks, before any is used."""
    return [ctypes.c_void_p(0x1000 * (i + 1)) for i in range(n)]


def test_loss_constant_matches_the_header():
    from agcn_b200 import _lib
    with open(os.path.join(ROOT, "include", "agcn_sgcll.h")) as f:
        defines = dict((k, int(v)) for k, v in re.findall(r"#define AGCN_LOSS_(\w+) (\d+)", f.read()))
    assert defines == {"SIGMOID_CE": 0, "SOFTMAX_CE": 1, "WEIGHTED_L2": 2}
    assert _lib.LOSS == {k.lower(): v for k, v in defines.items()}


def _descs():
    from agcn_b200 import _lib
    return (_lib.Desc * 2)(_lib.Desc(75, 64, 3, 0, 0, 0, 1, _lib.SAVE_FOR_BACKWARD),
                           _lib.Desc(64, 64, 3, 0, 0, 0, 1, _lib.SAVE_FOR_BACKWARD))


def test_stack_create_accepts_weighted_l2_and_rejects_unknown_kinds():
    from agcn_b200 import _lib
    lib = _lib.lib()
    offs = (ctypes.c_int64 * 14)(*range(14))
    stack = ctypes.c_void_p()
    assert lib.agcn_stack_create(_descs(), 2, 64, 1, 2, offs, ctypes.byref(stack)) == 0
    assert stack
    lib.agcn_stack_destroy(stack)
    for kind in (3, -1):
        stack = ctypes.c_void_p()
        assert lib.agcn_stack_create(_descs(), 2, 64, 1, kind, offs, ctypes.byref(stack)) == AGCN_ERR_INVALID
        assert "unknown loss_kind" in _last_error()
        assert not stack


def test_head_calls_check_their_arguments_for_weighted_l2():
    from agcn_b200 import _lib
    lib = _lib.lib()
    plan, H, dW, db, hW, hb, tg, w, out, loss, work, dH, g0, g1, g2, g3 = _fake(16)
    stream = ctypes.c_void_p(0)

    def predict(plan, tg, w, loss, kind=2, Fm=64, Nt=1):
        return lib.agcn_head_predict(plan, H, dW, db, hW, hb, tg, w, 1.0, kind, 64, Fm, Nt, out, loss, work, 1 << 20,
                                     stream)

    assert predict(None, None, None, None) == AGCN_ERR_INVALID
    assert "head_predict" in _last_error() and "null pointer" in _last_error()
    assert predict(None, tg, w, None) == AGCN_ERR_INVALID
    assert "all NULL or all set" in _last_error()
    assert predict(None, None, w, loss) == AGCN_ERR_INVALID
    assert "all NULL or all set" in _last_error()
    assert predict(plan, tg, w, loss, kind=3) == AGCN_ERR_INVALID
    assert "unknown loss_kind" in _last_error()
    # kind 2 passes the kind check (and, unlike the multitask classifier, takes an odd Nt): the size check comes next
    assert predict(plan, tg, w, loss, Fm=16) == AGCN_ERR_INVALID
    assert "unsupported sizes" in _last_error()

    def loss_grad(plan, kind=2, Fm=64, Nt=1):
        return lib.agcn_head_loss_grad_ex(plan, H, dW, db, hW, hb, tg, w, 1.0, kind, 64, Fm, Nt, loss, dH, g0, g1, g2,
                                          g3, work, 1 << 20, stream)

    assert loss_grad(None) == AGCN_ERR_INVALID
    assert "null pointer" in _last_error()
    assert loss_grad(plan, kind=3) == AGCN_ERR_INVALID
    assert "unknown loss_kind" in _last_error()
    assert loss_grad(plan, Fm=16) == AGCN_ERR_INVALID
    assert "unsupported sizes" in _last_error()


def test_stack_predict_checks_its_arguments_for_weighted_l2():
    from agcn_b200 import _lib
    lib = _lib.lib()
    offs = (ctypes.c_int64 * 14)(*range(14))
    stack = ctypes.c_void_p()
    _lib.check(lib.agcn_stack_create(_descs(), 2, 64, 1, _lib.LOSS["weighted_l2"], offs, ctypes.byref(stack)))
    try:
        X, L, tg, w, params, out, loss, work = _fake(8)
        stream = ctypes.c_void_p(0)

        def call(plan, tg, w, loss):
            return lib.agcn_stack_predict(stack, plan, X, L, tg, w, 1.0, params, out, loss, work, 1 << 20, stream)

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


def test_regressor_has_one_output_per_task_and_no_class_probabilities():
    from agcn_b200.simple_agcn import SimpleAGCNStep
    model = SimpleAGCNStep(75, (64, 128, 128, 64), 256, 3, 3, 8, device="cpu", loss="weighted_l2")
    assert model.Nt == 3 and tuple(model.head_W.shape) == (256, 3) and tuple(model.head_b.shape) == (3,)
    with pytest.raises(ValueError, match="no class probabilities"):
        model.predict_proba(None, None, None)
    with pytest.raises(ValueError):
        SimpleAGCNStep(75, (64, 128, 128, 64), 256, 3, 3, 8, device="cpu", loss="weighted_l1")


def test_synthetic_regression_labels():
    from agcn_b200.simple_agcn import synthetic_labels
    y, w = synthetic_labels(2000, 7, 5, "cpu", "weighted_l2")
    assert y.shape == w.shape == (2000, 7) and y.dtype == w.dtype == torch.float32
    assert set(np.unique(w.numpy()).tolist()) == {0.0, 1.0}
    assert 0.08 <= float((w == 0).float().mean()) <= 0.12
    assert abs(float(y.mean())) < 0.05 and abs(float(y.std()) - 1.0) < 0.05
    y2, w2 = synthetic_labels(2000, 7, 5, "cpu", "weighted_l2")
    assert torch.equal(y, y2) and torch.equal(w, w2)


def test_oracle_weighted_l2_and_its_closed_form_gradient():
    g = torch.Generator().manual_seed(1)
    B, T = 9, 4
    x = torch.randn(B, T, generator=g, dtype=torch.float64, requires_grad=True)
    y = torch.randn(B, T, generator=g, dtype=torch.float64)
    w = torch.rand(B, T, generator=g, dtype=torch.float64)
    w[0, 1] = 0.0
    scale = 1.0 / B
    loss = RO.weighted_l2(x, y, w, scale)
    want = sum(float((w[b, t] * (x[b, t] - y[b, t])) ** 2) for b in range(B) for t in range(T)) * scale
    assert abs(float(loss) - want) <= 1e-12 * want
    loss.backward()
    closed = RO.weighted_l2_grad(x.detach(), y, w, scale)
    assert torch.allclose(x.grad, closed, rtol=1e-12, atol=0)
    assert float(closed[0, 1]) == 0.0
    # the weight enters squared: halving every weight quarters the loss
    assert abs(float(RO.weighted_l2(x.detach(), y, w * 0.5, scale)) - 0.25 * float(loss)) <= 1e-12 * float(loss)


def test_oracle_head_values_are_the_linear_head_on_the_gathered_molecules():
    g = torch.Generator().manual_seed(2)
    Fh, Fm, T = 16, 32, 3
    H = [torch.randn(n, Fh, generator=g, dtype=torch.float64) for n in (3, 7, 11)]
    p = {"dense_W": torch.randn(Fh, Fm, generator=g, dtype=torch.float64) * 0.05,
         "dense_b": torch.randn(Fm, generator=g, dtype=torch.float64) * 0.02,
         "head_W": torch.randn(Fm, T, generator=g, dtype=torch.float64),
         "head_b": torch.randn(T, generator=g, dtype=torch.float64)}
    x = RO.head_values(H, p)
    mol = np.tanh(np.stack([(h.numpy() @ p["dense_W"].numpy() + p["dense_b"].numpy()).sum(0) for h in H]))
    assert x.shape == (3, T)
    assert np.allclose(x.numpy(), mol @ p["head_W"].numpy() + p["head_b"].numpy(), rtol=0, atol=1e-12)
