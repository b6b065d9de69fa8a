"""The node-list stack (agcn_stack_create_nodes) over node topologies other than ResAGCNStep's default layout.

The stack runner derives three pieces of topology-dependent machinery from the node list: the two gradient buffers of
the backward pass (which BlockEnd keeps its dpre alive, when dH[i-1] gets a second contribution and is copied into the
other buffer, how Reslap gradients flow back through dLall), the activation and L_all slots of prediction (reused once
their last reader has run), and the GEMM engines a BlockEnd's products take at its widths and batch size.  A wrong
liveness bound or a missing accumulate gives wrong numbers without any error, so every topology below is checked:

  1. loss and every gradient against the fp64 oracle (tests/residual_oracle.py, ReLU masks injected); every BlockEnd
     weight and every beta of a Reslap node with a src has a non-zero gradient;
  2. stack == autograd (the layer classes), bit for bit;
  3. the training arena (and the flat gradient buffer) filled with NaN bytes before the call: the same loss and
     gradients, bit for bit -- no buffer is read before it is written or accumulated into instead of overwritten;
  4. prediction: stack == autograd bit for bit and against the oracle; evaluate's loss == the training loss bit for
     bit; the same with the prediction arena filled with NaN bytes (the slots of agcn_stack_create_nodes).

Node notation: R = SGC_LL_Reslap, S = plain SGC_LL, BE = BlockEnd; node(src).
"""
import pytest
import torch

import predict_oracle as PO
import regression_oracle as RO
import residual_oracle as RES
from oracle import sgcll_oracle as O
from residual_topologies import N_FEAT, TOPOLOGIES, topology_model, widths
from util_cases import TOL, make_batch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
SCALAR_TOL = 2e-4   # dalpha / dbeta: sums with cancellation over every Laplacian entry (DESIGN.md section 6)
@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)     # the layer classes draw their glorot weights from the global generator


def _inputs(B=None, sizes=None, seed=1235):
    import agcn_b200
    if sizes is None:
        X, L, n = O.synthetic_molecule_batch(B, 132, seed=seed)
    else:
        X, L, n = make_batch(sizes, N_FEAT, max(sizes), seed=seed, kind="tox")
    batch = agcn_b200.GraphBatch(n, X.shape[1], device=DEV)
    return X, L, n, batch, batch.pack_nodes(torch.from_numpy(X).to(DEV)), batch.pack_lap(torch.from_numpy(L).to(DEV))


def _model(spec, B, n_tasks, loss, lap, mg, engine="stack"):
    from agcn_b200 import BlockEnd
    model = topology_model(spec, final_feature_n=256, n_tasks=n_tasks, K=3, batch_size=B, device=DEV, laplacian=lap,
                           metric_grad=mg, loss=loss, engine=engine, seed=11)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        # bias / alpha / beta / dense_b / head_b off their initial values so every gradient path is live
        for l in model.layers:
            if isinstance(l, BlockEnd):
                continue
            l.vars["bias"].copy_((torch.randn(l.vars["bias"].shape, generator=g) * 0.05).to(DEV))
            l.vars["alpha"].fill_(0.7)
            if "beta" in l.vars:
                l.vars["beta"].fill_(0.6)
            if lap == "paper":
                l.vars["weight"].mul_(0.3)   # keeps the learned metric out of fp32 denormals (test_gpu_network.py)
        model.dense_b.copy_((torch.randn(model.dense_b.shape, generator=g) * 0.02).to(DEV))
        model.head_b.copy_((torch.randn(model.head_b.shape, generator=g) * 0.05).to(DEV))
        model.dense_W.mul_(0.02)     # unsaturated GraphGatherMol tanh: the 1e-4 budget of test_gpu_network.py
    return model


def _labels(B, n_tasks, loss):
    from agcn_b200.simple_agcn import synthetic_labels
    y, w = synthetic_labels(B, n_tasks, 7, DEV, loss)
    return y, w * (0.5 + torch.rand(w.shape, generator=torch.Generator().manual_seed(3)).to(DEV))


def _acts(model):
    from agcn_b200 import BlockEnd
    from agcn_b200.operators import activations
    return ["linear" if isinstance(l, BlockEnd) and l.activation is activations.linear else "relu"
            for l in model.layers]


def _oracle_params(model, grad=True):
    nodes = [{k: v.detach().double().cpu().clone().requires_grad_(grad) for k, v in l.vars.items()}
             for l in model.layers]
    head = {k: getattr(model, k).detach().double().cpu().clone().requires_grad_(grad)
            for k in ("dense_W", "dense_b", "head_W", "head_b")}
    return nodes, head


def _relu_masks(model, Xd, Ld, batch):
    """Which outputs the CUDA path finds positive, node by node, as ResAGCNStep._body runs the layer classes."""
    from agcn_b200 import BlockEnd, SGC_LL_Reslap
    from agcn_b200.batch import PackedLaplacians, PackedNodes
    x = {'node_features': PackedNodes(Xd, batch), 'original_laplacian': PackedLaplacians(Ld, batch),
         'data_slice': None, 'lap_slice': None, '_batch': batch}
    masks, outs, lall = [], [], {}
    with torch.no_grad():
        for i, (layer, src) in enumerate(zip(model.layers, model.srcs)):
            if isinstance(layer, BlockEnd):
                out = layer(dict(x, block_outputs=outs[src]))
            elif isinstance(layer, SGC_LL_Reslap):
                out, _, _, lall[i] = layer(dict(x, res_lap=lall[src] if src >= 0 else []))
            else:
                out, _, _ = layer(x)
            masks.append((out.data > 0).cpu())
            outs.append(out)
            x = dict(x, node_features=out)
    return masks


def _split(model, flat):
    out, off = [], 0
    for p in model.params:
        out.append(flat[off:off + p.numel()])
        off += p.numel()
    return out


def _names(model):
    names = ["node%d.%s" % (i, k) for i, l in enumerate(model.layers) for k in l.vars]
    return names + ["dense_W", "dense_b", "head_W", "head_b"]


def _oracle_grads(model, nodes, head):
    parts = []
    for l, p in zip(model.layers, nodes):
        for k in l.vars:
            parts.append((torch.zeros_like(p[k]) if p[k].grad is None else p[k].grad).reshape(-1))
    return parts + [head[k].grad.reshape(-1) for k in ("dense_W", "dense_b", "head_W", "head_b")]


def _stack_step(model, Xd, Ld, batch, y, w, poison):
    """loss_and_grads on the stack engine with the arena and the gradient buffer zeroed, or filled with 0xFF bytes."""
    model._ensure_arena(batch)
    model._arena.fill_(0xFF if poison else 0)
    model.flat_grad.fill_(float("nan") if poison else 0.0)
    loss = float(model.loss_and_grads(Xd, Ld, batch, y, w))
    torch.cuda.synchronize()
    return loss, model.flat_grad.detach().clone()


def _stack_predict(model, Xd, Ld, batch, y, w, poison):
    """(predictions, evaluate's loss) on the stack engine with the prediction arena zeroed, or filled with 0xFF."""
    model._predict(Xd, Ld, batch)                       # sizes the arena
    model._pred_arena.fill_(0xFF if poison else 0)
    p, loss = model.evaluate(Xd, Ld, batch, y, w)
    p_only = model.predict(Xd, Ld, batch) if model.loss_kind == "weighted_l2" else model.predict_proba(Xd, Ld, batch)
    torch.cuda.synchronize()
    assert torch.equal(p, p_only), "evaluate's predictions differ from predict's"
    return p.clone(), float(loss)


CASES = [
    # name, topology, batch (molecule count, or explicit sizes), n_tasks, loss, laplacian, metric_grad
    ("block1", "block1", 48, 12, "sigmoid_ce", "reference_literal", "reference"),
    ("xres_is_x", "xres_is_x", 40, 10, "softmax_ce", "reference_literal", "reference"),
    ("xres_is_x_paper_full", "xres_is_x", 32, 12, "sigmoid_ce", "paper", "full"),
    ("be_after_be", "be_after_be", 48, 5, "weighted_l2", "reference_literal", "reference"),
    ("be_first", "be_first", 48, 12, "sigmoid_ce", "reference_literal", "reference"),
    ("long_range", "long_range", 40, 10, "softmax_ce", "reference_literal", "reference"),
    ("two_chains", "two_chains", 48, 5, "weighted_l2", "reference_literal", "reference"),
    ("mixed_plain", "mixed_plain", 48, 12, "sigmoid_ce", "reference_literal", "reference"),
    ("widths", "widths", 64, 12, "sigmoid_ce", "reference_literal", "reference"),
    # R = 26 < 32 rows: the BlockEnd products leave the tensor cores
    ("widths_small_batch", "widths", (4, 9, 6, 7), 5, "weighted_l2", "reference_literal", "reference"),
]


@pytest.mark.parametrize("name,topo,B,n_tasks,loss_kind,lap,mg", CASES, ids=[c[0] for c in CASES])
def test_topology_matches_oracle_autograd_and_poisoned_arenas(name, topo, B, n_tasks, loss_kind, lap, mg):
    spec = TOPOLOGIES[topo]
    X, L, n, batch, Xd, Ld = _inputs(sizes=B) if isinstance(B, tuple) else _inputs(B)
    B = len(n)
    y, w = _labels(B, n_tasks, loss_kind)
    model = _model(spec, B, n_tasks, loss_kind, lap, mg)
    assert [s for s in model.srcs] == [x[3] for x in widths(spec)]
    acts = _acts(model)
    X64, L64 = torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64)

    # ---- 1. the training step against the fp64 oracle
    nodes, head = _oracle_params(model)
    masks = _relu_masks(model, Xd, Ld, batch)
    loss_o = RES.res_agcn_loss(X64, L64, n, nodes, model.srcs, head, y.double().cpu(), w.double().cpu(), B, 3,
                               loss_kind, lap, mg, masks, acts)
    loss_o.backward()
    loss_o = float(loss_o.detach())
    grads_o = _oracle_grads(model, nodes, head)
    loss, g_stack = _stack_step(model, Xd, Ld, batch, y, w, poison=False)
    assert abs(loss - loss_o) <= TOL * abs(loss_o), (loss, loss_o)
    names = _names(model)
    worst = {}
    for nm, a, b in zip(names, _split(model, g_stack.cpu()), grads_o):
        worst[nm] = O.rel_err(a, b) if float(b.abs().max()) > 0 else float(a.abs().max())
    print(name, "loss %.9g, oracle %.9g" % (loss, loss_o))
    print(name, "worst gradient %.1e (alpha / beta %.1e)" % (
        max(v for k, v in worst.items() if not k.endswith((".alpha", ".beta"))),
        max(v for k, v in worst.items() if k.endswith((".alpha", ".beta")))))
    bad = {k: v for k, v in worst.items() if not v <= (SCALAR_TOL if k.endswith((".alpha", ".beta")) else TOL)}
    assert not bad, "gradient mismatch vs oracle: %s" % {k: "%.1e" % v for k, v in bad.items()}
    live = ["node%d.weight" % i for i, x in enumerate(widths(spec)) if x[0] == "BE"]
    live += ["node%d.beta" % i for i, x in enumerate(widths(spec)) if x[0] == "R" and x[3] >= 0]
    for nm, a in zip(names, _split(model, g_stack.cpu())):
        if nm in live:
            assert float(a.abs().max()) > 0, "%s has a zero gradient" % nm

    # ---- 2. the layer classes under autograd: the same numbers, bit for bit
    model.flat_grad.zero_()
    model.engine = "autograd"
    loss_a = float(model.loss_and_grads(Xd, Ld, batch, y, w))
    torch.cuda.synchronize()
    model.engine = "stack"
    assert loss_a == loss
    assert torch.equal(model.flat_grad, g_stack), "stack and autograd engines disagree"

    # ---- 3. NaN bytes in the arena and the gradient buffer change nothing
    loss_p, g_p = _stack_step(model, Xd, Ld, batch, y, w, poison=True)
    assert loss_p == loss and torch.equal(g_p, g_stack), "the training step read a buffer it had not written"

    # ---- 4. prediction
    p_stack, loss_e = _stack_predict(model, Xd, Ld, batch, y, w, poison=False)
    assert loss_e == loss, "evaluate's loss differs from loss_and_grads' loss"
    p_poison, loss_ep = _stack_predict(model, Xd, Ld, batch, y, w, poison=True)
    assert loss_ep == loss and torch.equal(p_poison, p_stack), "prediction read a slot it had not written"
    model.engine = "autograd"
    p_a, loss_a = model.evaluate(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    model.engine = "stack"
    assert float(loss_a) == loss and torch.equal(p_a, p_stack), "stack and autograd predictions disagree"
    nodes, head = _oracle_params(model, grad=False)
    H = RES.res_agcn_features(X64, L64, n, nodes, model.srcs, 3, lap, mg, acts=acts)
    if loss_kind == "weighted_l2":
        err = O.rel_err(p_stack.cpu(), RO.head_values(H, head))
        print(name, "values: max-abs error / max-abs reference %.1e" % err)
        assert err <= TOL
    else:
        err = O.rel_err(p_stack.cpu(), PO.head_predict(H, head, loss_kind))
        print(name, "probabilities: max-abs error / max-abs reference %.1e" % err)
        assert err <= 1e-5

