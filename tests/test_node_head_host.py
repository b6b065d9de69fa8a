"""The per-node classification head (loss="node_softmax_ce") without a GPU: its loss constant in the C ABI and the
Python binding, the argument checks of the node-head calls and of the kind in agcn_stack_create(_nodes) (they reject
bad calls before anything touches the device), SimpleAGCNStep's flat-buffer layout for the head, the synthetic node
labels, and the fp64 reference against its closed-form gradient."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import node_head_oracle as NHO

AGCN_ERR_INVALID = -1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from agcn_b200 import _lib
    return _lib


def _last_error():
    return _lib().lib().agcn_last_error().decode()


def _fake(n):
    """Distinct non-NULL addresses: the calls below must fail on their argument checks, before any is used."""
    return [ctypes.c_void_p(0x1000 * (i + 1)) for i in range(n)]


def _descs():
    L = _lib()
    return (L.Desc * 2)(L.Desc(3, 64, 3, 0, 0, 0, 1, L.SAVE_FOR_BACKWARD), L.Desc(64, 64, 3, 0, 0, 0, 1,
                                                                                   L.SAVE_FOR_BACKWARD))


def _offs(dense=(-1, -1)):
    """5 per layer for the two layers of _descs, then dense_W, dense_b, head_W, head_b."""
    return (ctypes.c_int64 * 14)(*(list(range(10)) + list(dense) + [10, 11]))


def test_node_loss_constant_matches_the_header():
    L = _lib()
    with open(os.path.join(ROOT, "include", "agcn_sgcll.h")) as f:
        defines = dict((k, int(v)) for k, v in re.findall(r"#define AGCN_PER_NODE_(\w+) (\d+)", f.read()))
    assert defines == {"SOFTMAX_CE": 4}
    assert L.NODE_LOSS == {"node_" + k.lower(): v for k, v in defines.items()}
    assert not set(L.NODE_LOSS.values()) & set(L.LOSS.values())
    assert L.loss_code("node_softmax_ce") == 4 and L.loss_code("softmax_ce") == 1
    with pytest.raises(ValueError):
        L.loss_code("node_sigmoid_ce")


def test_unknown_kinds_are_still_rejected_everywhere():
    L = _lib()
    lib = L.lib()
    for kind in (3, -1, 7):
        stack = ctypes.c_void_p()
        assert lib.agcn_stack_create(_descs(), 2, 64, 4, kind, _offs((10, 11)), ctypes.byref(stack)) == AGCN_ERR_INVALID
        assert "unknown loss_kind" in _last_error() and not stack
        nodes = (L.StackNode * 1)(L.StackNode(L.NODE["sgcll"], _descs()[0], -1))
        offs = (ctypes.c_int64 * 9)(*range(9))
        assert lib.agcn_stack_create_nodes(nodes, 1, 64, 4, kind, offs, ctypes.byref(stack)) == AGCN_ERR_INVALID
        assert "unknown loss_kind" in _last_error()


def test_graph_head_calls_reject_the_node_kind_and_name_the_node_head_calls():
    lib = _lib().lib()
    plan, H, dW, db, hW, hb, tg, w, out, loss, work, dH, g0, g1, g2, g3 = _fake(16)
    stream = ctypes.c_void_p(0)
    assert lib.agcn_head_predict(plan, H, dW, db, hW, hb, tg, w, 1.0, 4, 64, 64, 4, out, loss, work, 1 << 20,
                                 stream) == AGCN_ERR_INVALID
    assert "agcn_node_head_predict" in _last_error()
    assert lib.agcn_head_loss_grad_ex(plan, H, dW, db, hW, hb, tg, w, 1.0, 4, 64, 64, 4, loss, dH, g0, g1, g2, g3,
                                      work, 1 << 20, stream) == AGCN_ERR_INVALID
    assert "agcn_node_head_loss_grad" in _last_error()


def test_node_head_calls_check_their_arguments():
    lib = _lib().lib()
    plan, H, hW, hb, tg, w, out, loss, work, dH, g0, g1 = _fake(12)
    stream = ctypes.c_void_p(0)

    def predict(plan, tg, w, loss, H=H, out=out, work=work, Fh=64, C=13):
        return lib.agcn_node_head_predict(plan, H, hW, hb, tg, w, 1.0, Fh, C, out, loss, work, 1 << 20, stream)

    assert predict(None, None, None, None) == AGCN_ERR_INVALID
    assert "node_head_predict" in _last_error() and "null pointer" in _last_error()
    for args in ((plan, tg, w, None), (plan, None, w, loss), (plan, tg, None, loss), (plan, tg, None, None)):
        assert predict(*args) == AGCN_ERR_INVALID
        assert "all NULL or all set" in _last_error()
    for kw in ({"H": None}, {"out": None}, {"work": None}):
        assert predict(plan, tg, w, loss, **kw) == AGCN_ERR_INVALID
        assert "null pointer" in _last_error()
    for Fh, C in ((0, 13), (64, 0)):
        assert predict(plan, tg, w, loss, Fh=Fh, C=C) == AGCN_ERR_INVALID
        assert "unsupported sizes" in _last_error()

    def loss_grad(*ptrs, Fh=64, C=13):
        return lib.agcn_node_head_loss_grad(*ptrs[:6], 1.0, Fh, C, *ptrs[6:], 1 << 20, stream)

    full = [plan, H, hW, hb, tg, w, loss, dH, g0, g1, work]
    for i in range(len(full)):
        ptrs = list(full)
        ptrs[i] = None
        assert loss_grad(*ptrs) == AGCN_ERR_INVALID
        assert "node_head_loss_grad: null pointer" in _last_error()
    for Fh, C in ((0, 13), (64, 0)):
        assert loss_grad(*full, Fh=Fh, C=C) == AGCN_ERR_INVALID
        assert "unsupported sizes" in _last_error()

    size = ctypes.c_size_t()
    for fn in (lib.agcn_node_head_workspace_bytes, lib.agcn_node_head_predict_workspace_bytes):
        assert fn(None, 64, 13, ctypes.byref(size)) == AGCN_ERR_INVALID
        assert fn(plan, 0, 13, ctypes.byref(size)) == AGCN_ERR_INVALID
        assert fn(plan, 64, 0, ctypes.byref(size)) == AGCN_ERR_INVALID
        assert fn(plan, 64, 13, None) == AGCN_ERR_INVALID
        assert "workspace_bytes: bad arguments" in _last_error()


def test_stack_create_takes_the_node_kind_only_without_the_dense_pair():
    L = _lib()
    lib = L.lib()
    kind = L.NODE_LOSS["node_softmax_ce"]
    stack = ctypes.c_void_p()
    assert lib.agcn_stack_create(_descs(), 2, 0, 13, kind, _offs(), ctypes.byref(stack)) == 0
    assert stack
    lib.agcn_stack_destroy(stack)
    stack = ctypes.c_void_p()
    assert lib.agcn_stack_create(_descs(), 2, 64, 13, kind, _offs(), ctypes.byref(stack)) == AGCN_ERR_INVALID
    assert "Fm must be 0" in _last_error() and not stack
    assert lib.agcn_stack_create(_descs(), 2, 0, 0, kind, _offs(), ctypes.byref(stack)) == AGCN_ERR_INVALID
    assert "Nt >= 1" in _last_error()
    for dense in ((10, -1), (-1, 10), (10, 11)):
        assert lib.agcn_stack_create(_descs(), 2, 0, 13, kind, _offs(dense), ctypes.byref(stack)) == AGCN_ERR_INVALID
        assert "offsets must be -1" in _last_error() and not stack
    # the graph heads keep their checks: Fm = 0 is still refused for them
    assert lib.agcn_stack_create(_descs(), 2, 0, 13, L.LOSS["softmax_ce"], _offs((10, 11)),
                                 ctypes.byref(stack)) == AGCN_ERR_INVALID
    assert "Fm and Nt must be positive" in _last_error()
    # the node-list form: a residual body
    nodes = (L.StackNode * 3)(L.StackNode(L.NODE["sgcll"], L.Desc(3, 64, 3, 1, 0, 0, 1, 0), -1),
                              L.StackNode(L.NODE["sgcll"], L.Desc(64, 64, 3, 1, 0, 0, 1, 0), 0),
                              L.StackNode(L.NODE["block_end"], L.Desc(64, 64, 0, 0, 0, 0, 1, 0), 0))
    offs = list(range(15)) + [-1, -1, 20, 21]
    assert lib.agcn_stack_create_nodes(nodes, 3, 0, 50, kind, (ctypes.c_int64 * 19)(*offs), ctypes.byref(stack)) == 0
    lib.agcn_stack_destroy(stack)
    offs[15] = 16
    stack = ctypes.c_void_p()
    assert lib.agcn_stack_create_nodes(nodes, 3, 0, 50, kind, (ctypes.c_int64 * 19)(*offs),
                                       ctypes.byref(stack)) == AGCN_ERR_INVALID
    assert "offsets must be -1" in _last_error()


@pytest.mark.parametrize("residual", [False, True], ids=["simple", "residual"])
def test_step_layout_and_flat_buffer_offsets(residual):
    from agcn_b200.residual_agcn import ResAGCNStep
    from agcn_b200.simple_agcn import SimpleAGCNStep
    base_cls = ResAGCNStep if residual else SimpleAGCNStep

    class Probe(base_cls):
        def _create_stack(self, offs):
            self.offs = list(offs)
            super(Probe, self)._create_stack(offs)

    filters = (64, 64, 64) if residual else (64, 128, 64)
    model = Probe(3, filters, 999, 13, 3, 4, device="cpu", loss="node_softmax_ce")
    assert model.Fm == 0 and model.Nt == 13 and model.dense_W is None and model.dense_b is None
    assert tuple(model.head_W.shape) == (64, 13) and tuple(model.head_b.shape) == (13,)
    assert float(model.head_W.detach().abs().max()) <= 0.02 and float(model.head_W.detach().std()) > 0
    n = len(model.layers)
    base = model.flat_params.flat.data_ptr()
    assert model.offs[5 * n:] == [-1, -1, (model.head_W.data_ptr() - base) // 4, (model.head_b.data_ptr() - base) // 4]
    assert model.params[-2:] == [model.head_W, model.head_b]
    # notify stage n covers head_W and head_b, and the stages tile the flat buffer
    a, b = model._stage_slices[n]
    assert (a, b) == (model.offs[5 * n + 2], model.n_parameters()) and b - a == 64 * 13 + 13
    assert model._stage_slices[0][0] == 0
    assert all(model._stage_slices[i][1] == model._stage_slices[i + 1][0] for i in range(n))
    # the body is drawn as for the other losses: same layer parameters for the same seed
    other = base_cls(3, filters, 256, 13, 3, 4, device="cpu", loss="softmax_ce")
    for la, lb in zip(model.layers, other.layers):
        for k in la.vars:
            assert torch.equal(la.vars[k], lb.vars[k])


def test_final_feature_n_is_ignored_and_unknown_losses_are_refused():
    from agcn_b200.simple_agcn import SimpleAGCNStep
    SimpleAGCNStep(3, (64,), 7, 5, 3, 4, device="cpu", loss="node_softmax_ce")      # 7 would be refused by a graph head
    with pytest.raises(ValueError):
        SimpleAGCNStep(3, (64,), 7, 5, 3, 4, device="cpu", loss="softmax_ce")
    with pytest.raises(ValueError):
        SimpleAGCNStep(3, (64,), 256, 5, 3, 4, device="cpu", loss="node_weighted_l2")


def test_synthetic_node_labels_point_clouds():
    from agcn_b200.synthetic import modelnet_like_batch, synthetic_node_labels, sydney_like_batch
    for X, _, n in (modelnet_like_batch(2, 256, seed=3), sydney_like_batch(6, 200, seed=4)):
        for C in (2, 13, 50):
            y, w = synthetic_node_labels(n, X, C, 9)
            R = int(n.sum())
            assert y.shape == (R, C) and w.shape == (R,) and y.dtype == w.dtype == np.float32
            assert np.array_equal(y.sum(1), np.ones(R, np.float32)) and set(np.unique(y).tolist()) == {0.0, 1.0}
            assert set(np.unique(w).tolist()) == {0.0, 1.0} and 0.05 <= float((w == 0).mean()) <= 0.15
            # the label is a function of the point's own xyz: the same point in another graph position gets it too
            rows = np.concatenate([X[g, :k] for g, k in enumerate(n)])
            lab = y.argmax(1)
            assert len(np.unique(lab)) >= min(C, 4)
            y2, w2 = synthetic_node_labels(n, X, C, 9)
            assert np.array_equal(y, y2) and np.array_equal(w, w2)
            assert not np.array_equal(w, synthetic_node_labels(n, X, C, 10)[1])
        # sector x band: with C = 4 (2 x 2) the label splits on the sign of atan2(z, x) and on the height median
        y4, _ = synthetic_node_labels(n, X, 4, 1)
        lab = y4.argmax(1)
        assert np.array_equal(lab // 2, (np.arctan2(rows[:, 2], rows[:, 0]) >= 0).astype(int))


def test_synthetic_node_labels_molecules():
    from agcn_b200.synthetic import molecule_batch, synthetic_node_labels
    X, _, n = molecule_batch(5, 40, seed=2)
    y, w = synthetic_node_labels(n, X, 7, 1)
    rows = np.concatenate([X[g, :k] for g, k in enumerate(n)])
    assert np.array_equal(y.argmax(1), rows[:, :44].argmax(1) % 7)
    assert w.shape == (int(n.sum()),)


def test_oracle_node_loss_and_its_closed_form_gradient():
    g = torch.Generator().manual_seed(4)
    R, C = 37, 13
    x = torch.randn(R, C, generator=g, dtype=torch.float64, requires_grad=True)
    y = torch.zeros(R, C, dtype=torch.float64)
    y[torch.arange(R), torch.randint(0, C, (R,), generator=g)] = 1.0
    w = (torch.rand(R, generator=g, dtype=torch.float64) >= 0.1).double() * (0.5 + torch.rand(R, generator=g,
                                                                                                  dtype=torch.float64))
    w[3] = 0.0
    scale = 1.0 / 5
    loss = NHO.node_softmax_ce(x, y, w, scale)
    want = sum(float(w[r]) * (float(torch.logsumexp(x[r], 0)) - float(x[r, int(y[r].argmax())])) for r in range(R))
    assert abs(float(loss) - want * scale) <= 1e-12 * abs(want)
    loss.backward()
    closed = NHO.node_ce_grad(x.detach(), y, w, scale)
    assert torch.allclose(x.grad, closed, rtol=1e-12, atol=1e-15)
    assert float(closed[3].abs().max()) == 0.0           # a masked node contributes nothing
    # the logits: H head_W + head_b over the concatenated graphs
    H = [torch.randn(k, 8, generator=g, dtype=torch.float64) for k in (3, 5)]
    W, b = torch.randn(8, C, generator=g, dtype=torch.float64), torch.randn(C, generator=g, dtype=torch.float64)
    assert torch.allclose(NHO.node_logits(H, W, b), torch.cat(H) @ W + b, rtol=0, atol=1e-12)
