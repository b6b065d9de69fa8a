"""The regression head of the SimpleAGCN stack (loss="weighted_l2": MultitaskGraphRegressor's one output per task and
weighted L2 loss) on the device:

  * the training step against the fp64 oracle network: the loss, every gradient of the flat buffer and the parameters
    after Adam, at the Delaney shape (B = 256, one task), with 12 tasks and fractional weights, at the C2 shape (B = 1024,
    617 tasks: several 64-column tiles of the output product) and with paper/full semantics; engine "stack" == engine
    "autograd" and CUDA-graph replay == eager launches, bit for bit;
  * the weights: halving every weight scales the loss by 1/4, and a zero weight removes its (b, t) from the loss and the
    gradients;
  * prediction: the values against the oracle, the evaluation loss bit-identical to the training loss, no state touched,
    stack == autograd, replay == eager, whole batch == four quarters;
  * ten steps on one batch lower the loss, reproducibly.
"""
import numpy as np
import pytest
import torch

import regression_oracle as RO
from oracle import network_oracle as NO
from oracle import sgcll_oracle as O
from util_cases import TOL

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
LOSS = "weighted_l2"


def _perturb(model, seed):
    """Bias / alpha / dense_b / head_b off their initial values so every gradient path is live (as test_gpu_network.py)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for l in model.layers:
            l.vars["bias"].copy_((torch.randn(l.vars["bias"].shape, generator=g) * 0.05).to(l.vars["bias"].device))
            l.vars["alpha"].fill_(0.7)
        model.dense_b.copy_((torch.randn(model.dense_b.shape, generator=g) * 0.02).to(model.dense_b.device))
        model.head_b.copy_((torch.randn(model.head_b.shape, generator=g) * 0.05).to(model.head_b.device))


def _inputs(B, seed=1235):
    import agcn_b200
    X, L, n = O.synthetic_molecule_batch(B, 132, seed=seed)
    batch = agcn_b200.GraphBatch(n, 132, device=DEV)
    return X, L, n, batch, batch.pack_nodes(torch.from_numpy(X).to(DEV)), batch.pack_lap(torch.from_numpy(L).to(DEV))


def _model(B, n_tasks, lap="reference_literal", mg="reference", dense_scale=1.0, seed=11):
    from agcn_b200.simple_agcn import SimpleAGCNStep
    model = SimpleAGCNStep(75, (64, 128, 128, 64), 256, n_tasks, 3, B, device=DEV, laplacian=lap, metric_grad=mg,
                           loss=LOSS, engine="stack", seed=seed)
    _perturb(model, 5)
    with torch.no_grad():
        model.dense_W.mul_(dense_scale)
        if lap == "paper":
            for l in model.layers:
                l.vars["weight"].mul_(0.3)    # keeps the learned metric out of fp32 denormals (test_gpu_network.py)
    return model


def _labels(B, n_tasks, fractional=False):
    from agcn_b200.simple_agcn import synthetic_labels
    y, w = synthetic_labels(B, n_tasks, 7, DEV, LOSS)
    if fractional:
        w = w * (0.5 + torch.rand(w.shape, generator=torch.Generator().manual_seed(3)).to(DEV))
    return y, w


def _oracle_params(model):
    layer_p = [{k: v.detach().double().cpu().clone().requires_grad_(True) for k, v in l.vars.items()}
               for l in model.layers]
    head_p = {k: getattr(model, k).detach().double().cpu().clone().requires_grad_(True)
              for k in ("dense_W", "dense_b", "head_W", "head_b")}
    return layer_p, head_p


def _flat_oracle_grad(layer_p, head_p):
    parts = []
    for p in layer_p:
        for k in ("weight", "bias", "M_L", "alpha"):
            g = p[k].grad
            parts.append((torch.zeros_like(p[k]) if g is None else g).reshape(-1))
    for k in ("dense_W", "dense_b", "head_W", "head_b"):
        parts.append(head_p[k].grad.reshape(-1))
    return parts


def _names(model):
    out = []
    for i in range(len(model.layers)):
        out += ["layer%d.%s" % (i, k) for k in ("weight", "bias", "M_L", "alpha")]
    return out + ["dense_W", "dense_b", "head_W", "head_b"]


def _split(model, flat):
    out, off = [], 0
    for p in model.params:
        out.append(flat[off:off + p.numel()])
        off += p.numel()
    return out


def _relu_masks(model, Xd, Ld, batch):
    """Which outputs the CUDA path finds positive, layer by layer (NO.simple_agcn_features)."""
    from agcn_b200.batch import PackedLaplacians, PackedNodes
    masks = []
    with torch.no_grad():
        xin = {'node_features': PackedNodes(Xd, batch), 'original_laplacian': PackedLaplacians(Ld, batch),
               'data_slice': None, 'lap_slice': None, '_batch': batch}
        for layer in model.layers:
            out, _, _ = layer(xin)
            masks.append((out.data > 0).cpu())
            xin = dict(xin, node_features=out)
    return masks


@pytest.fixture(scope="module")
def c2():
    """The C2-shaped batch (B = 1024 molecules) shared by the tests below."""
    return _inputs(1024)


# Tolerances as tests/test_gpu_network.py: 1e-3 for the network as initialised (GraphGatherMol's tanh of a sum over the
# atoms is saturated and amplifies the rounding of the layers ~100x), 1e-4 with DenseMol's weights scaled by 0.02.
CASES = [
    # name, B, n_tasks, fractional weights, laplacian, metric_grad, dense_scale, tolerance
    ("delaney_T1_literal", 256, 1, False, "reference_literal", "reference", 1.0, 1e-3),
    ("delaney_T1_literal_unsaturated", 256, 1, False, "reference_literal", "reference", 0.02, TOL),
    ("T12_fractional_weights_unsaturated", 256, 12, True, "reference_literal", "reference", 0.02, TOL),
    ("C2_T617_literal_unsaturated", 1024, 617, False, "reference_literal", "reference", 0.02, TOL),
    ("T12_paper_full", 256, 12, True, "paper", "full", 1.0, 1e-3),
]


@pytest.mark.parametrize("name,B,n_tasks,fractional,lap,mg,dense_scale,tol", CASES, ids=[c[0] for c in CASES])
def test_regression_step_matches_oracle_network(name, B, n_tasks, fractional, lap, mg, dense_scale, tol):
    X, L, n, batch, Xd, Ld = _inputs(B)
    y, w = _labels(B, n_tasks, fractional)
    model = _model(B, n_tasks, lap, mg, dense_scale)
    assert model.Nt == n_tasks and tuple(model.head_W.shape) == (256, n_tasks)
    layer_p, head_p = _oracle_params(model)
    p_before = model.flat_params.flat.detach().clone()
    masks = _relu_masks(model, Xd, Ld, batch)

    X64, L64 = torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64)
    loss_o = RO.simple_agcn_loss(X64, L64, n, layer_p, head_p, y.double().cpu(), w.double().cpu(), B, 3, lap, mg, masks)
    loss_o.backward()
    grads_o = _flat_oracle_grad(layer_p, head_p)

    loss = model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    g_stack = model.flat_grad.detach().clone()
    print(name, "loss %.9g, oracle %.9g" % (float(loss), float(loss_o)))
    assert abs(float(loss) - float(loss_o)) <= TOL * abs(float(loss_o)), (float(loss), float(loss_o))
    worst = {}
    for nm, a, b in zip(_names(model), _split(model, g_stack.cpu()), grads_o):
        worst[nm] = O.rel_err(a, b) if float(b.abs().max()) > 0 else float(a.abs().max())
    print(name, {k: "%.1e" % v for k, v in worst.items()})
    bad = {k: v for k, v in worst.items() if not v <= tol}
    assert not bad, "gradient mismatch vs oracle network: %s" % bad

    # the drop-in path (layer classes + autograd): the same numbers, bit for bit
    model.flat_grad.zero_()
    model.engine = "autograd"
    loss_a = model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    model.engine = "stack"
    assert float(loss_a) == float(loss)
    assert torch.equal(model.flat_grad, g_stack), "stack and autograd engines disagree"

    # CUDA-graph replay == eager launches, bit for bit
    model.flat_grad.zero_()
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        model.loss_and_grads(Xd, Ld, batch, y, w)
    model.flat_grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(model.flat_grad, g_stack), "CUDA-graph replay differs from eager launches"
    assert float(model._loss) == float(loss)
    del graph

    # Adam: two steps against tf.train.AdamOptimizer's rule
    p_o = p_before.double().cpu()
    m_o = torch.zeros_like(p_o)
    v_o = torch.zeros_like(p_o)
    for t in (1, 2):
        model.apply_adam()
        p_o, m_o, v_o = NO.adam_tf(p_o, g_stack.double().cpu(), m_o, v_o, t, lr=model.lr, eps=model.epsilon)
    torch.cuda.synchronize()
    assert int(model.adam_step) == 2
    assert O.rel_err(model.flat_params.flat.detach().cpu(), p_o) <= 1e-6
    assert O.rel_err((model.flat_params.flat.detach() - p_before).cpu(), p_o - p_before.double().cpu()) <= 1e-4


def test_weights_enter_squared_and_zero_weights_mask_labels():
    B, T = 256, 12
    X, L, n, batch, Xd, Ld = _inputs(B)
    y, w = _labels(B, T, fractional=True)
    model = _model(B, T)
    loss = float(model.loss_and_grads(Xd, Ld, batch, y, w))
    grads = model.flat_grad.detach().clone()
    loss_half = float(model.loss_and_grads(Xd, Ld, batch, y, w * 0.5))
    torch.cuda.synchronize()
    print("loss %.9g, with halved weights %.9g (x4 = %.9g)" % (loss, loss_half, 4 * loss_half))
    assert abs(4.0 * loss_half - loss) <= 1e-6 * loss

    # a zero weight: its target does not matter, bit for bit
    zero = torch.rand(w.shape, generator=torch.Generator().manual_seed(9)).to(DEV) < 0.3
    w0 = torch.where(zero, torch.zeros_like(w), w)
    loss0 = float(model.loss_and_grads(Xd, Ld, batch, y, w0))
    grads0 = model.flat_grad.detach().clone()
    y_moved = torch.where(zero, y + 5.0 * torch.randn(y.shape, generator=torch.Generator().manual_seed(4)).to(DEV), y)
    loss0_moved = float(model.loss_and_grads(Xd, Ld, batch, y_moved, w0))
    torch.cuda.synchronize()
    assert int(zero.sum()) > 0 and not torch.equal(y_moved, y)
    assert loss0_moved == loss0
    assert torch.equal(model.flat_grad, grads0)
    assert loss0 != loss and not torch.equal(grads0, grads)
    # the values the device predicts, and the weighted-L2 terms in fp64: zeroed terms left the loss
    x = model.predict(Xd, Ld, batch).double()
    want = float(RO.weighted_l2(x, y.double(), w0.double(), 1.0 / B))
    assert abs(loss0 - want) <= 1e-5 * want


# The values are compared as they are, not through a softmax that compresses them: in the network as initialised the
# fp32 rounding of GraphGatherMol's saturated sums reaches x at ~2e-5 of its largest value (1.8e-5 at T = 1, 2.1e-5 at
# T = 617 on a B200 at 1000 W), so that network is held to the layer budget and the unsaturated one (DenseMol x 0.02,
# as in the parity test) to 1e-5.
PREDICT_CASES = [
    # name, B, n_tasks, dense_scale, tolerance
    ("delaney_T1", 256, 1, 1.0, TOL),
    ("delaney_T1_unsaturated", 256, 1, 0.02, 1e-5),
    ("C2_T617", 1024, 617, 1.0, TOL),
    ("C2_T617_unsaturated", 1024, 617, 0.02, 1e-5),
]


@pytest.mark.parametrize("name,B,n_tasks,dense_scale,tol", PREDICT_CASES, ids=[c[0] for c in PREDICT_CASES])
def test_predict_values_match_oracle_and_evaluate_loss_is_the_training_loss(c2, name, B, n_tasks, dense_scale, tol):
    X, L, n, batch, Xd, Ld = c2 if B == 1024 else _inputs(B)
    y, w = _labels(B, n_tasks, fractional=True)
    model = _model(B, n_tasks, dense_scale=dense_scale)
    x = model.predict(Xd, Ld, batch)
    torch.cuda.synchronize()
    assert x.shape == (B, n_tasks) and x.dtype == torch.float32
    with pytest.raises(ValueError):
        model.predict_proba(Xd, Ld, batch)
    layer_p = [{k: v.detach().double().cpu() for k, v in l.vars.items()} for l in model.layers]
    head_p = {k: getattr(model, k).detach().double().cpu() for k in ("dense_W", "dense_b", "head_W", "head_b")}
    H = NO.simple_agcn_features(torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64), n, layer_p,
                                3)
    want = RO.head_values(H, head_p)
    err = O.rel_err(x.cpu(), want)
    print(name, "values: max-abs error / max-abs reference %.1e" % err)
    assert err <= tol

    # evaluate's loss is loss_and_grads' loss, bit for bit, with both engines
    loss_t = float(model.loss_and_grads(Xd, Ld, batch, y, w))
    x_e, loss_e = model.evaluate(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    print("training loss %.9g, evaluate loss %.9g" % (loss_t, float(loss_e)))
    assert float(loss_e) == loss_t, "evaluate's loss differs from loss_and_grads' loss"
    assert torch.equal(x_e, x)
    model.engine = "autograd"
    x_a, loss_a = model.evaluate(Xd, Ld, batch, y, w)
    assert torch.equal(model.predict(Xd, Ld, batch), x), "stack and autograd engines disagree"
    model.engine = "stack"
    assert float(loss_a) == loss_t and torch.equal(x_a, x)

    # parameters, gradients and Adam state: bit-unchanged by predict / evaluate
    model.apply_adam()
    model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    state = [t.detach().clone() for t in (model.flat_grad, model.flat_params.flat, model.adam_m, model.adam_v,
                                          model.adam_step)]
    model.predict(Xd, Ld, batch)
    model.evaluate(Xd, Ld, batch, y, w)
    model.engine = "autograd"
    model.evaluate(Xd, Ld, batch, y, w)
    model.engine = "stack"
    torch.cuda.synchronize()
    for before, now in zip(state, (model.flat_grad, model.flat_params.flat, model.adam_m, model.adam_v,
                                   model.adam_step)):
        assert torch.equal(before, now)


def test_predict_graph_replay_matches_eager_and_the_batch_split(c2):
    import agcn_b200
    X, L, n, batch, Xd, Ld = c2
    model = _model(1024, 617)
    eager = model.predict(Xd, Ld, batch).clone()
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        model.predict(Xd, Ld, batch)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        replayed = model.predict(Xd, Ld, batch)
    replayed.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(replayed, eager), "CUDA-graph replay differs from eager launches"
    del graph

    parts = []
    for q in range(4):
        sl = slice(256 * q, 256 * (q + 1))
        b = agcn_b200.GraphBatch(n[sl], X.shape[1], device=DEV)
        parts.append(model.predict(b.pack_nodes(torch.from_numpy(X[sl]).to(DEV)),
                                   b.pack_lap(torch.from_numpy(L[sl]).to(DEV)), b))
    quarters = torch.cat(parts, 0)
    torch.cuda.synchronize()
    diff = float((eager - quarters).abs().max())
    print("whole batch vs four quarters: max abs difference %.3e, bit-identical: %s"
          % (diff, bool(torch.equal(eager, quarters))))
    assert torch.equal(eager, quarters)


def test_regression_step_decreases_loss_and_is_reproducible():
    """Ten full steps (loss_and_grads + Adam) on one batch: the loss goes down, and a second model with the same seed
    follows the same trajectory bit for bit."""
    from agcn_b200.simple_agcn import SimpleAGCNStep, synthetic_labels
    B, T = 128, 3
    X, L, n, batch, Xd, Ld = _inputs(B, seed=77)
    y, w = synthetic_labels(B, T, 3, DEV, LOSS)
    traj = []
    for rep in range(2):
        model = SimpleAGCNStep(75, (64, 128, 128, 64), 256, T, 3, B, device=DEV, seed=5, loss=LOSS)
        losses = [float(model.step(Xd, Ld, batch, y, w)) for _ in range(10)]
        traj.append(losses)
        print("losses", losses)
        assert np.isfinite(losses).all() and losses[-1] < losses[0]
    assert traj[0] == traj[1]
