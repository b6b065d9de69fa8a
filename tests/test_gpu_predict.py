"""Prediction with the SimpleAGCN stack (SimpleAGCNStep.predict_proba / predict / evaluate, agcn_stack_predict,
agcn_head_predict) on the device:

  * probabilities against the fp64 oracle network for the C1 / C2 molecule heads (literal and paper/full semantics), the
    single-task softmax head and a C3-shaped point-cloud batch (graphs of 1024 nodes: the row-tiled forward path);
  * the evaluation loss is bit-identical to the training step's loss, and prediction leaves the parameters, gradients
    and Adam state alone;
  * engine "stack" == engine "autograd" and CUDA-graph replay == eager launches, bit for bit;
  * a batch predicted whole or in quarters gives the same probabilities;
  * a prediction costs less arena and fewer launches than a training step.
"""
import numpy as np
import pytest
import torch

from oracle import network_oracle as NO
from oracle import sgcll_oracle as O
from predict_oracle import head_predict
from util_cases import TOL

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _perturb(model, seed):
    """Bias / alpha / dense_b / head_b off their initial values (as tests/test_gpu_network.py does)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for l in model.layers:
            l.vars["bias"].copy_((torch.randn(l.vars["bias"].shape, generator=g) * 0.05).to(l.vars["bias"].device))
            l.vars["alpha"].fill_(0.7)
        model.dense_b.copy_((torch.randn(model.dense_b.shape, generator=g) * 0.02).to(model.dense_b.device))
        model.head_b.copy_((torch.randn(model.head_b.shape, generator=g) * 0.05).to(model.head_b.device))


def _inputs(gen, B):
    import agcn_b200
    from agcn_b200 import synthetic
    if gen == "points":
        X, L, n = synthetic.modelnet_like_batch(B, 1024, seed=1236)
    else:
        X, L, n = O.synthetic_molecule_batch(B, 132, seed=1235)
    batch = agcn_b200.GraphBatch(n, X.shape[1], device=DEV)
    return X, L, n, batch, batch.pack_nodes(torch.from_numpy(X).to(DEV)), batch.pack_lap(torch.from_numpy(L).to(DEV))


def _model(F, B, n_tasks, loss, lap="reference_literal", mg="reference", engine="stack"):
    from agcn_b200.simple_agcn import SimpleAGCNStep
    model = SimpleAGCNStep(F, (64, 128, 128, 64), 256, n_tasks, 3, B, device=DEV, laplacian=lap, metric_grad=mg,
                           loss=loss, engine=engine, seed=11)
    _perturb(model, 5)
    if lap == "paper":
        with torch.no_grad():
            for l in model.layers:
                l.vars["weight"].mul_(0.3)    # keeps the learned metric out of fp32 denormals (test_gpu_network.py)
    return model


def _labels(B, n_tasks, loss):
    from agcn_b200.simple_agcn import synthetic_labels
    tg, w = synthetic_labels(B, n_tasks, 7, DEV, loss)
    return tg, w * (0.5 + torch.rand(w.shape, generator=torch.Generator().manual_seed(3)).to(DEV))


@pytest.fixture(scope="module")
def c2():
    """The C2 batch (B = 1024 molecules, 617 tasks) shared by the tests below."""
    return _inputs("molecules", 1024)


CASES = [
    # name, input kind, B, n_tasks, loss, laplacian, metric_grad
    ("C1_literal", "molecules", 256, 12, "sigmoid_ce", "reference_literal", "reference"),
    ("C2_literal", "molecules", 1024, 617, "sigmoid_ce", "reference_literal", "reference"),
    ("C1_paper_full", "molecules", 256, 12, "sigmoid_ce", "paper", "full"),
    ("softmax_head", "molecules", 96, 40, "softmax_ce", "reference_literal", "reference"),
    ("C3_points", "points", 4, 40, "softmax_ce", "reference_literal", "reference"),
]


@pytest.mark.parametrize("name,gen,B,n_tasks,loss,lap,mg", CASES, ids=[c[0] for c in CASES])
def test_predict_proba_matches_oracle_and_engines_agree(name, gen, B, n_tasks, loss, lap, mg):
    X, L, n, batch, Xd, Ld = _inputs(gen, B)
    model = _model(X.shape[2], B, n_tasks, loss, lap, mg)
    probs = model.predict_proba(Xd, Ld, batch)
    labels = model.predict(Xd, Ld, batch)
    torch.cuda.synchronize()
    want_shape = (B, n_tasks, 2) if loss == "sigmoid_ce" else (B, n_tasks)
    assert probs.shape == want_shape and probs.dtype == torch.float32
    assert labels.shape == want_shape[:-1] and labels.dtype == torch.int64
    assert torch.equal(labels, probs.argmax(-1))

    layer_p = [{k: v.detach().double().cpu() for k, v in l.vars.items()} for l in model.layers]
    head_p = {k: getattr(model, k).detach().double().cpu() for k in ("dense_W", "dense_b", "head_W", "head_b")}
    H = NO.simple_agcn_features(torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64), n, layer_p,
                                3, lap, mg)
    want = head_predict(H, head_p, loss)
    err = O.rel_err(probs.cpu(), want)
    print(name, "probabilities: max-abs error / max-abs reference %.1e" % err)
    assert err <= TOL
    assert float((probs.double().sum(-1) - 1).abs().max()) <= 1e-5

    # the drop-in path: layer classes under no_grad + functional.head_predict
    model.engine = "autograd"
    probs_a = model.predict_proba(Xd, Ld, batch)
    torch.cuda.synchronize()
    assert torch.equal(probs_a, probs), "stack and autograd engines disagree"


@pytest.mark.parametrize("loss", ["sigmoid_ce", "softmax_ce"])
def test_evaluate_loss_is_the_training_loss_and_leaves_the_state_alone(c2, loss):
    if loss == "sigmoid_ce":
        X, L, n, batch, Xd, Ld = c2
        B, n_tasks = 1024, 617
    else:
        B, n_tasks = 96, 40
        X, L, n, batch, Xd, Ld = _inputs("molecules", B)
    tg, w = _labels(B, n_tasks, loss)
    model = _model(75, B, n_tasks, loss)
    loss_t = float(model.loss_and_grads(Xd, Ld, batch, tg, w))
    probs, loss_e = model.evaluate(Xd, Ld, batch, tg, w)
    torch.cuda.synchronize()
    print(loss, "training loss %.9g, evaluate loss %.9g" % (loss_t, float(loss_e)))
    assert float(loss_e) == loss_t, "evaluate's loss differs from loss_and_grads' loss"
    assert torch.equal(probs, model.predict_proba(Xd, Ld, batch))
    model.engine = "autograd"
    _, loss_a = model.evaluate(Xd, Ld, batch, tg, w)
    model.engine = "stack"
    assert float(loss_a) == loss_t

    # parameters, gradients and Adam state: bit-unchanged by predict_proba / evaluate
    model.apply_adam()
    model.loss_and_grads(Xd, Ld, batch, tg, w)
    torch.cuda.synchronize()
    state = [t.detach().clone() for t in (model.flat_grad, model.flat_params.flat, model.adam_m, model.adam_v,
                                          model.adam_step)]
    model.predict_proba(Xd, Ld, batch)
    model.evaluate(Xd, Ld, batch, tg, w)
    model.engine = "autograd"
    model.evaluate(Xd, Ld, batch, tg, w)
    torch.cuda.synchronize()
    for before, now in zip(state, (model.flat_grad, model.flat_params.flat, model.adam_m, model.adam_v,
                                   model.adam_step)):
        assert torch.equal(before, now)


def test_predict_proba_graph_replay_matches_eager(c2):
    X, L, n, batch, Xd, Ld = c2
    model = _model(75, 1024, 617, "sigmoid_ce")
    eager = model.predict_proba(Xd, Ld, batch).clone()
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        model.predict_proba(Xd, Ld, batch)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        replayed = model.predict_proba(Xd, Ld, batch)
    replayed.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(replayed, eager), "CUDA-graph replay differs from eager launches"
    del graph


def test_predict_is_independent_of_the_batch_split(c2):
    import agcn_b200
    X, L, n, batch, Xd, Ld = c2
    model = _model(75, 1024, 617, "sigmoid_ce")
    whole = model.predict_proba(Xd, Ld, batch)
    parts = []
    for q in range(4):
        sl = slice(256 * q, 256 * (q + 1))
        b = agcn_b200.GraphBatch(n[sl], X.shape[1], device=DEV)
        parts.append(model.predict_proba(b.pack_nodes(torch.from_numpy(X[sl]).to(DEV)),
                                         b.pack_lap(torch.from_numpy(L[sl]).to(DEV)), b))
    quarters = torch.cat(parts, 0)
    torch.cuda.synchronize()
    diff = float((whole - quarters).abs().max())
    print("whole batch vs four quarters: max abs difference %.3e, bit-identical: %s"
          % (diff, bool(torch.equal(whole, quarters))))
    assert diff <= 1e-6


def test_predict_costs_less_than_a_training_step(c2):
    import ctypes

    from agcn_b200 import _lib
    X, L, n, batch, Xd, Ld = c2
    model = _model(75, 1024, 617, "sigmoid_ce")
    tg, w = _labels(1024, 617, "sigmoid_ce")
    lib = _lib.lib()
    pred_b, train_b = ctypes.c_size_t(), ctypes.c_size_t()
    _lib.check(lib.agcn_stack_predict_workspace_bytes(model._stack, batch.handle, ctypes.byref(pred_b)))
    _lib.check(lib.agcn_stack_workspace_bytes(model._stack, batch.handle, ctypes.byref(train_b)))
    model.predict_proba(Xd, Ld, batch)                 # arenas allocated outside the counted calls
    model.loss_and_grads(Xd, Ld, batch, tg, w)
    c0 = _lib.launch_count()
    model.predict_proba(Xd, Ld, batch)
    c1 = _lib.launch_count()
    model.loss_and_grads(Xd, Ld, batch, tg, w)
    c2_ = _lib.launch_count()
    torch.cuda.synchronize()
    print("C2 arena: predict %d bytes, training step %d bytes; launches: predict %d, loss_and_grads %d"
          % (pred_b.value, train_b.value, c1 - c0, c2_ - c1))
    assert pred_b.value < train_b.value
    assert c1 - c0 < c2_ - c1
