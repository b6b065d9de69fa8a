"""The per-node classification head (loss="node_softmax_ce"): one part label per node, trained and predicted in one
call by the SGC-LL stack, against the fp64 reference of tests/node_head_oracle.py (ReLU masks injected as in
tests/test_gpu_network.py).

Shapes: C1 molecules (F = 75), 100-node clouds (the ShapeNet part-segmentation shape, F = 3), two 1024-point clouds
(ModelNet shape) and a ragged Sydney-shape batch; C in {2, 13, 50, 64, 100} (odd, not a multiple of 4, above one warp
and one 64-column tile); both semantics modes; one ResAGCNStep case.  Each case checks:
  * the loss and every gradient against the oracle;
  * engine "stack" == engine "autograd", bit for bit; CUDA-graph replay == eager launches, bit for bit;
  * the same loss, gradients, probabilities and evaluation loss with both arenas filled with NaN bytes;
  * the probabilities against the oracle; evaluate's loss == the training loss, bit for bit;
  * predict / evaluate leave parameters, gradients and Adam state untouched;
  * a batch predicted whole == the same batch predicted in quarters (batches of four graphs or more);
  * ten Adam steps lower the loss, two runs with one seed agree, and step_graphed follows step bit for bit.
"""
import numpy as np
import pytest
import torch

import node_head_oracle as NHO
from oracle import sgcll_oracle as O
from util_cases import TOL

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
SCALAR_TOL = 2e-4   # dalpha / dbeta: sums with cancellation over every Laplacian entry (DESIGN.md section 6)


def _batch(shape):
    """(X, L, n_nodes) in the wire layout."""
    from agcn_b200 import synthetic as S
    if shape == "C1":
        return O.synthetic_molecule_batch(64, 132, seed=1235)
    if shape == "shapenet":
        return S.modelnet_like_batch(16, 100, seed=21)
    if shape == "modelnet":
        return S.modelnet_like_batch(2, 1024, seed=22)
    if shape == "sydney":
        return S.sydney_like_batch(12, 300, seed=23)
    raise ValueError(shape)


# name, shape, C, laplacian, metric_grad, residual
CASES = [
    ("C1_C13_literal", "C1", 13, "reference_literal", "reference", False),
    ("shapenet_C50_literal", "shapenet", 50, "reference_literal", "reference", False),
    ("shapenet_C2_paper_full", "shapenet", 2, "paper", "full", False),
    ("modelnet_C64_literal", "modelnet", 64, "reference_literal", "reference", False),
    ("sydney_C100_literal", "sydney", 100, "reference_literal", "reference", False),
    ("res_shapenet_C13_literal", "shapenet", 13, "reference_literal", "reference", True),
]


def _model(X, n, C, lap, mg, residual, seed=11):
    from agcn_b200 import BlockEnd
    from agcn_b200.residual_agcn import ResAGCNStep
    from agcn_b200.simple_agcn import SimpleAGCNStep
    F, B = X.shape[2], len(n)
    if residual:
        model = ResAGCNStep(F, (64, 64, 64), 0, C, 3, B, device=DEV, laplacian=lap, metric_grad=mg,
                            loss="node_softmax_ce", seed=seed)
    else:
        model = SimpleAGCNStep(F, (64, 128, 64), 0, C, 3, B, device=DEV, laplacian=lap, metric_grad=mg,
                               loss="node_softmax_ce", seed=seed)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        # bias / alpha / head_b off their initial values so every gradient path is live
        for l in model.layers:
            if isinstance(l, BlockEnd):
                continue
            l.vars["bias"].copy_((torch.randn(l.vars["bias"].shape, generator=g) * 0.05).to(DEV))
            l.vars["alpha"].fill_(0.7)
            if lap == "paper":          # keep the learned metric's distances in fp32 range (tests/test_gpu_network.py)
                l.vars["weight"].mul_(0.3)
        model.head_b.copy_((torch.randn(model.head_b.shape, generator=g) * 0.05).to(DEV))
        model.head_W.mul_(20.0)         # a softmax far from uniform
    return model


def _inputs(X, L, n):
    import agcn_b200
    batch = agcn_b200.GraphBatch(n, X.shape[1], device=DEV)
    return batch, batch.pack_nodes(torch.from_numpy(X).to(DEV)), batch.pack_lap(torch.from_numpy(L).to(DEV))


def _labels(n, X, C, seed=7):
    from agcn_b200.synthetic import synthetic_node_labels
    y, w = synthetic_node_labels(n, X, C, seed)
    w = w * (0.5 + np.random.default_rng(3).random(w.shape, dtype=np.float32))     # non-trivial weights
    return torch.from_numpy(y).to(DEV), torch.from_numpy(w).to(DEV)


def _relu_masks(model, Xd, Ld, batch):
    """Which outputs the CUDA path finds positive, node by node (the layer classes, wired as the model's _body)."""
    from agcn_b200 import BlockEnd, SGC_LL_Reslap
    from agcn_b200.batch import PackedLaplacians, PackedNodes
    x = {'node_features': PackedNodes(Xd, batch), 'original_laplacian': PackedLaplacians(Ld, batch),
         'data_slice': None, 'lap_slice': None, '_batch': batch}
    srcs = getattr(model, "srcs", [-1] * len(model.layers))
    outs, lall, masks = [], {}, []
    with torch.no_grad():
        for i, (layer, src) in enumerate(zip(model.layers, srcs)):
            if isinstance(layer, BlockEnd):
                out = layer(dict(x, block_outputs=outs[src]))
            elif isinstance(layer, SGC_LL_Reslap):
                out, _, _, lall[i] = layer(dict(x, res_lap=lall[src] if src >= 0 else []))
            else:
                out, _, _ = layer(x)
            outs.append(out)
            masks.append((out.data > 0).cpu())
            x = dict(x, node_features=out)
    return masks


def _oracle(model, X, L, n, y, w, lap, mg, masks, grad=True):
    nodes = [{k: v.detach().double().cpu().clone().requires_grad_(grad) for k, v in l.vars.items()}
             for l in model.layers]
    head = {k: getattr(model, k).detach().double().cpu().clone().requires_grad_(grad) for k in ("head_W", "head_b")}
    srcs = getattr(model, "srcs", [-1] * len(model.layers))
    loss, x = NHO.node_agcn_loss(torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64), n, nodes,
                                 srcs, head, y.double().cpu(), w.double().cpu(), model.global_batch, 3, lap, mg, masks)
    names, grads = [], []
    if grad:
        loss.backward()
        for i, (l, p) in enumerate(zip(model.layers, nodes)):
            for k in l.vars:
                names.append("node%d.%s" % (i, k))
                grads.append(p[k].grad if p[k].grad is not None else torch.zeros_like(p[k]))
        names += ["head_W", "head_b"]
        grads += [head["head_W"].grad, head["head_b"].grad]
    return loss.detach(), torch.softmax(x.detach(), 1), names, grads


def _split(model, flat):
    out, off = [], 0
    for p in model.params:
        out.append(flat[off:off + p.numel()].reshape(p.shape))
        off += p.numel()
    return out


@pytest.mark.parametrize("name,shape,C,lap,mg,residual", CASES, ids=[c[0] for c in CASES])
def test_node_head(name, shape, C, lap, mg, residual):
    import agcn_b200
    X, L, n = _batch(shape)
    batch, Xd, Ld = _inputs(X, L, n)
    R = int(n.sum())
    y, w = _labels(n, X, C)
    model = _model(X, n, C, lap, mg, residual)

    # ---- loss and every gradient against the fp64 oracle
    masks = _relu_masks(model, Xd, Ld, batch)
    loss_o, probs_o, names, grads_o = _oracle(model, X, L, n, y, w, lap, mg, masks)
    loss = model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    g_stack = model.flat_grad.detach().clone()
    loss_t = float(loss)
    print(name, "R %d, loss %.9g, oracle %.9g" % (R, loss_t, float(loss_o)))
    assert abs(loss_t - float(loss_o)) <= TOL * abs(float(loss_o)), (loss_t, float(loss_o))
    worst = {}
    for nm, a, b in zip(names, _split(model, g_stack.cpu()), grads_o):
        worst[nm] = O.rel_err(a, b) if float(b.abs().max()) > 0 else float(a.abs().max())
    print(name, {k: "%.1e" % v for k, v in worst.items()})
    bad = {k: v for k, v in worst.items()
           if not v <= (max(TOL, SCALAR_TOL) if k.endswith((".alpha", ".beta")) else TOL)}
    assert not bad, "gradient mismatch vs oracle: %s" % bad
    assert float(g_stack.abs().max()) > 0 and all(float(t.abs().max()) > 0 for t in _split(model, g_stack)[-2:])

    # ---- the layer classes and node_head_loss under autograd: the same numbers, bit for bit
    model.flat_grad.zero_()
    model.engine = "autograd"
    loss_a = model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    model.engine = "stack"
    assert float(loss_a) == loss_t
    assert torch.equal(model.flat_grad, g_stack), "stack and autograd engines disagree"

    # ---- CUDA-graph replay == eager launches, bit for bit
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
    assert float(model._loss) == loss_t
    del graph

    # ---- prediction: probabilities against the oracle, evaluate's loss == the training loss, stack == autograd
    probs = model.predict_proba(Xd, Ld, batch)
    labels = model.predict(Xd, Ld, batch)
    torch.cuda.synchronize()
    assert probs.shape == (R, C) and labels.shape == (R,) and labels.dtype == torch.int64
    assert torch.equal(labels, probs.argmax(-1))
    err = O.rel_err(probs.cpu(), probs_o)
    print(name, "probabilities: max-abs error / max-abs reference %.1e" % err)
    # per-node logits reach tens of nats here (head_W scaled by 20, unnormalised cloud coordinates): a probability
    # carries the logits' absolute fp32 error, so the layer's 1e-4 budget applies rather than the graph heads' 1e-5
    assert err <= TOL
    p_e, loss_e = model.evaluate(Xd, Ld, batch, y, w, scale=1.0 / model.global_batch)
    assert float(loss_e) == loss_t, "evaluate's loss differs from loss_and_grads' loss"
    assert torch.equal(p_e, probs)
    model.engine = "autograd"
    p_a, loss_a = model.evaluate(Xd, Ld, batch, y, w, scale=1.0 / model.global_batch)
    model.engine = "stack"
    assert float(loss_a) == loss_t and torch.equal(p_a, probs), "stack and autograd engines disagree"
    padded = batch.unpack_nodes(probs)
    assert padded.shape == (len(n), X.shape[1], C) and torch.equal(padded[0, :int(n[0])], probs[:int(n[0])])

    # ---- NaN bytes in both arenas (and the gradient buffer) change nothing
    model._arena.fill_(0xFF)
    model._pred_arena.fill_(0xFF)
    model.flat_grad.fill_(float("nan"))
    assert float(model.loss_and_grads(Xd, Ld, batch, y, w)) == loss_t
    p_n, loss_n = model.evaluate(Xd, Ld, batch, y, w, scale=1.0 / model.global_batch)
    torch.cuda.synchronize()
    assert torch.equal(model.flat_grad, g_stack), "stale arena bytes reached the gradients"
    assert torch.equal(p_n, probs) and float(loss_n) == loss_t, "stale arena bytes reached the prediction"

    # ---- parameters, gradients and Adam state: bit-unchanged by predict / evaluate
    model.apply_adam()
    model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    state = [t.detach().clone() for t in (model.flat_grad, model.flat_params.flat, model.adam_m, model.adam_v,
                                          model.adam_step)]
    model.predict(Xd, Ld, batch)
    model.evaluate(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    for before, now in zip(state, (model.flat_grad, model.flat_params.flat, model.adam_m, model.adam_v,
                                   model.adam_step)):
        assert torch.equal(before, now)

    # ---- the batch whole == the batch in quarters (the head is row by row; the body is per graph)
    if len(n) >= 4:
        whole = model.predict_proba(Xd, Ld, batch)
        parts, q = [], len(n) // 4
        for k in range(4):
            sl = slice(q * k, q * (k + 1) if k < 3 else len(n))
            b = agcn_b200.GraphBatch(n[sl], X.shape[1], device=DEV)
            parts.append(model.predict_proba(b.pack_nodes(torch.from_numpy(X[sl]).to(DEV)),
                                             b.pack_lap(torch.from_numpy(L[sl]).to(DEV)), b))
        quarters = torch.cat(parts, 0)
        print(name, "whole vs quarters: max abs difference %.3e" % float((whole - quarters).abs().max()))
        assert torch.equal(whole, quarters)

    # ---- ten Adam steps lower the loss; two runs with one seed agree; step_graphed follows step bit for bit
    runs = []
    for graphed in (False, False, True):
        m = _model(X, n, C, lap, mg, residual, seed=5)
        fn = m.step_graphed if graphed else m.step
        losses = [float(fn(Xd, Ld, batch, y, w)) for _ in range(10)]
        torch.cuda.synchronize()
        runs.append((losses, m.flat_params.flat.detach().clone()))
    print(name, "losses", runs[0][0])
    assert np.isfinite(runs[0][0]).all() and runs[0][0][-1] < runs[0][0][0]
    for losses, params in runs[1:]:
        assert losses == runs[0][0] and torch.equal(params, runs[0][1])
