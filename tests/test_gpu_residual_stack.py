"""The residual AGCN stack (agcn_stack_create_nodes: SGC_LL_Reslap layers chained through L_all, BlockEnd residual
blocks; agcn_b200.residual_agcn.ResAGCNStep) on the device:

  * the training step against the fp64 oracle (tests/residual_oracle.py, ReLU masks of every layer and BlockEnd output
    injected): loss and every gradient of the flat buffer at C1 and C2 in literal mode, as initialised and unsaturated,
    paper/full, a weighted-L2 and a softmax head; every beta and BlockEnd weight gradient is non-zero; stack ==
    autograd and CUDA-graph replay == eager, bit for bit; Adam after two steps;
  * prediction: probabilities against the oracle, evaluate's loss == the training loss bit for bit, no state touched,
    stack == autograd, replay == eager, whole C2 batch == four quarters;
  * ten steps lower the loss reproducibly; step_graphed == step over batches of changing composition;
  * the notify stages cover the flat buffer exactly once, in backward order;
  * a plain SGC_LL stack built from a node list == agcn_stack_create, bit for bit and launch for launch.
"""
import ctypes

import numpy as np
import pytest
import torch

import predict_oracle as PO
import residual_oracle as RES
from oracle import network_oracle as NO
from oracle import sgcll_oracle as O
from util_cases import TOL

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
SCALAR_TOL = 2e-4   # dalpha / dbeta: sums with cancellation over every Laplacian entry (DESIGN.md section 6)


def _inputs(B, seed=1235, nmax=None):
    import agcn_b200
    X, L, n = O.synthetic_molecule_batch(B, 132, seed=seed)
    if nmax is not None:
        n = np.minimum(n, nmax).astype(np.int32)
    batch = agcn_b200.GraphBatch(n, 132, device=DEV)
    return X, L, n, batch, batch.pack_nodes(torch.from_numpy(X).to(DEV)), batch.pack_lap(torch.from_numpy(L).to(DEV))


def _model(B, n_tasks, loss="sigmoid_ce", lap="reference_literal", mg="reference", dense_scale=1.0, seed=11,
           engine="stack"):
    from agcn_b200 import BlockEnd
    from agcn_b200.residual_agcn import ResAGCNStep
    model = ResAGCNStep(75, (64, 64, 64, 64, 64), 256, n_tasks, 3, B, device=DEV, laplacian=lap, metric_grad=mg,
                        loss=loss, engine=engine, seed=seed)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        # bias / alpha / beta / dense_b / head_b off their initial values so every gradient path is live
        for l in model.layers:
            if isinstance(l, BlockEnd):
                continue
            l.vars["bias"].copy_((torch.randn(l.vars["bias"].shape, generator=g) * 0.05).to(DEV))
            l.vars["alpha"].fill_(0.7)
            l.vars["beta"].fill_(0.6)
        model.dense_b.copy_((torch.randn(model.dense_b.shape, generator=g) * 0.02).to(DEV))
        model.head_b.copy_((torch.randn(model.head_b.shape, generator=g) * 0.05).to(DEV))
        model.dense_W.mul_(dense_scale)
        if lap == "paper":
            for l in model.layers:
                if not isinstance(l, BlockEnd):
                    l.vars["weight"].mul_(0.3)   # keeps the learned metric out of fp32 denormals (test_gpu_network.py)
    return model


def _labels(B, n_tasks, loss):
    from agcn_b200.simple_agcn import synthetic_labels
    y, w = synthetic_labels(B, n_tasks, 7, DEV, loss)
    return y, w * (0.5 + torch.rand(w.shape, generator=torch.Generator().manual_seed(3)).to(DEV))


def _oracle_params(model, grad=True):
    nodes = [{k: v.detach().double().cpu().clone().requires_grad_(grad) for k, v in l.vars.items()}
             for l in model.layers]
    head = {k: getattr(model, k).detach().double().cpu().clone().requires_grad_(grad)
            for k in ("dense_W", "dense_b", "head_W", "head_b")}
    return nodes, head


def _names_and_oracle_grads(model, nodes, head):
    names, parts = [], []
    for i, (l, p) in enumerate(zip(model.layers, nodes)):
        for k, v in l.vars.items():
            names.append("node%d.%s" % (i, k))
            parts.append((torch.zeros_like(p[k]) if p[k].grad is None else p[k].grad).reshape(-1))
    for k in ("dense_W", "dense_b", "head_W", "head_b"):
        names.append(k)
        parts.append(head[k].grad.reshape(-1))
    return names, parts


def _split(model, flat):
    out, off = [], 0
    for p in model.params:
        out.append(flat[off:off + p.numel()])
        off += p.numel()
    return out


def _relu_masks(model, Xd, Ld, batch):
    """Which outputs the CUDA path finds positive, node by node (residual_oracle.res_agcn_features)."""
    from agcn_b200 import BlockEnd
    from agcn_b200.batch import PackedLaplacians, PackedNodes
    x = {'node_features': PackedNodes(Xd, batch), 'original_laplacian': PackedLaplacians(Ld, batch),
         'data_slice': None, 'lap_slice': None, '_batch': batch}
    masks, outs, lall = [], [], {}
    with torch.no_grad():
        for i, (layer, src) in enumerate(zip(model.layers, model.srcs)):
            if isinstance(layer, BlockEnd):
                out = layer(dict(x, block_outputs=outs[src]))
            else:
                out, _, _, lall[i] = layer(dict(x, res_lap=lall[src] if src >= 0 else []))
            masks.append((out.data > 0).cpu())
            outs.append(out)
            x = dict(x, node_features=out)
    return masks


@pytest.fixture(scope="module")
def c2():
    return _inputs(1024)


# Tolerances as tests/test_gpu_network.py: 1e-3 for the network as initialised (GraphGatherMol's saturated tanh
# amplifies the rounding of the layers ~100x), 1e-4 with DenseMol's weights scaled by 0.02; the scalar gradients at 2e-4.
CASES = [
    # name, B, n_tasks, loss, laplacian, metric_grad, dense_scale, tolerance
    ("C1_literal", 256, 12, "sigmoid_ce", "reference_literal", "reference", 1.0, 1e-3),
    ("C1_literal_unsaturated", 256, 12, "sigmoid_ce", "reference_literal", "reference", 0.02, TOL),
    ("C2_literal", 1024, 617, "sigmoid_ce", "reference_literal", "reference", 1.0, 1e-3),
    ("C2_literal_unsaturated", 1024, 617, "sigmoid_ce", "reference_literal", "reference", 0.02, TOL),
    ("C1_paper_full", 256, 12, "sigmoid_ce", "paper", "full", 1.0, 1e-3),
    ("weighted_l2_unsaturated", 256, 12, "weighted_l2", "reference_literal", "reference", 0.02, TOL),
    ("softmax_unsaturated", 96, 40, "softmax_ce", "reference_literal", "reference", 0.02, TOL),
]


@pytest.mark.parametrize("name,B,n_tasks,loss_kind,lap,mg,dense_scale,tol", CASES, ids=[c[0] for c in CASES])
def test_residual_step_matches_oracle(c2, name, B, n_tasks, loss_kind, lap, mg, dense_scale, tol):
    X, L, n, batch, Xd, Ld = c2 if B == 1024 else _inputs(B)
    y, w = _labels(B, n_tasks, loss_kind)
    model = _model(B, n_tasks, loss_kind, lap, mg, dense_scale)
    nodes, head = _oracle_params(model)
    p_before = model.flat_params.flat.detach().clone()
    masks = _relu_masks(model, Xd, Ld, batch)

    X64, L64 = torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64)
    loss_o = RES.res_agcn_loss(X64, L64, n, nodes, model.srcs, head, y.double().cpu(), w.double().cpu(), B, 3,
                               loss_kind, lap, mg, masks)
    loss_o.backward()
    names, grads_o = _names_and_oracle_grads(model, nodes, head)

    loss = model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    g_stack = model.flat_grad.detach().clone()
    print(name, "loss %.9g, oracle %.9g" % (float(loss), float(loss_o)))
    assert abs(float(loss) - float(loss_o)) <= TOL * abs(float(loss_o)), (float(loss), float(loss_o))
    worst = {}
    for nm, a, b in zip(names, _split(model, g_stack.cpu()), grads_o):
        worst[nm] = O.rel_err(a, b) if float(b.abs().max()) > 0 else float(a.abs().max())
    print(name, {k: "%.1e" % v for k, v in worst.items()})
    bad = {k: v for k, v in worst.items()
           if not v <= (max(tol, SCALAR_TOL) if k.endswith((".alpha", ".beta")) else tol)}
    assert not bad, "gradient mismatch vs oracle: %s" % bad
    for nm, a in zip(names, _split(model, g_stack.cpu())):
        if nm.endswith(".beta") and nm != "node0.beta" or nm in ("node3.weight", "node6.weight"):
            assert float(a.abs().max()) > 0, "%s has a zero gradient" % nm

    # the layer classes under autograd: the same numbers, bit for bit
    model.flat_grad.zero_()
    model.engine = "autograd"
    loss_a = model.loss_and_grads(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    model.engine = "stack"
    assert float(loss_a) == float(loss)
    assert torch.equal(model.flat_grad, g_stack), "stack and autograd engines disagree"

    # CUDA-graph replay == eager launches, bit for bit
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


def test_residual_predict(c2):
    import agcn_b200
    X, L, n, batch, Xd, Ld = c2
    B, T = 1024, 617
    y, w = _labels(B, T, "sigmoid_ce")
    model = _model(B, T, dense_scale=0.02)
    probs = model.predict_proba(Xd, Ld, batch)
    torch.cuda.synchronize()
    assert probs.shape == (B, T, 2)
    nodes, head = _oracle_params(model, grad=False)
    H = RES.res_agcn_features(torch.tensor(X, dtype=torch.float64), torch.tensor(L, dtype=torch.float64), n, nodes,
                              model.srcs, 3)
    err = O.rel_err(probs.cpu(), PO.head_predict(H, head, "sigmoid_ce"))
    print("probabilities: max-abs error / max-abs reference %.1e" % err)
    assert err <= 1e-5

    # evaluate's loss is loss_and_grads' loss, bit for bit; stack == autograd
    loss_t = float(model.loss_and_grads(Xd, Ld, batch, y, w))
    p_e, loss_e = model.evaluate(Xd, Ld, batch, y, w)
    torch.cuda.synchronize()
    assert float(loss_e) == loss_t, "evaluate's loss differs from loss_and_grads' loss"
    assert torch.equal(p_e, probs)
    model.engine = "autograd"
    p_a, loss_a = model.evaluate(Xd, Ld, batch, y, w)
    model.engine = "stack"
    assert float(loss_a) == loss_t and torch.equal(p_a, probs), "stack and autograd engines disagree"

    # parameters, gradients and Adam state: bit-unchanged by predict / evaluate
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

    # CUDA-graph replay == eager; the batch whole == the batch in quarters
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
    parts = []
    for q in range(4):
        sl = slice(256 * q, 256 * (q + 1))
        b = agcn_b200.GraphBatch(n[sl], X.shape[1], device=DEV)
        parts.append(model.predict_proba(b.pack_nodes(torch.from_numpy(X[sl]).to(DEV)),
                                         b.pack_lap(torch.from_numpy(L[sl]).to(DEV)), b))
    assert torch.equal(eager, torch.cat(parts, 0))


def test_residual_step_decreases_loss_is_reproducible_and_graphed_matches_eager():
    from agcn_b200.residual_agcn import ResAGCNStep
    from agcn_b200.simple_agcn import synthetic_labels
    B = 128
    X, L, n, batch, Xd, Ld = _inputs(B, seed=77)
    y, w = synthetic_labels(B, 12, 3, DEV)
    traj = []
    for rep in range(2):
        model = ResAGCNStep(device=DEV, batch_size=B, seed=5)
        losses = [float(model.step(Xd, Ld, batch, y, w)) for _ in range(10)]
        traj.append(losses)
        print("losses", losses)
        assert np.isfinite(losses).all() and losses[-1] < losses[0]
    assert traj[0] == traj[1]

    # step_graphed == step over batches of changing composition (another set of size buckets in the third)
    batches = [_inputs(96, seed=s, nmax=m)[3:] for s, m in ((1, None), (2, None), (3, 40))]
    y, w = synthetic_labels(96, 12, 3, DEV)
    runs = []
    for graphed in (False, True):
        model = ResAGCNStep(device=DEV, batch_size=96, seed=5)
        losses = []
        for k in (0, 1, 0, 2, 1, 0):
            b, Xb, Lb = batches[k]
            losses.append(float((model.step_graphed if graphed else model.step)(Xb, Lb, b, y, w)))
        torch.cuda.synchronize()
        runs.append((losses, model.flat_params.flat.detach().clone(), model.step_graph_updates))
    assert np.isfinite(runs[0][0]).all()
    assert runs[0][0] == runs[1][0]
    assert torch.equal(runs[0][1], runs[1][1])
    assert runs[1][2] >= 2


def test_notify_stages_cover_the_flat_buffer_in_backward_order():
    from agcn_b200 import _lib
    from agcn_b200.batch import _ptr, _stream_ptr
    B = 64
    X, L, n, batch, Xd, Ld = _inputs(B)
    y, w = _labels(B, 12, "sigmoid_ce")
    model = _model(B, 12)
    model._ensure_arena(batch)
    stages = []
    cb = _lib.NOTIFY_FN(lambda _u, stage, _s: stages.append(int(stage)))
    _lib.check(_lib.lib().agcn_stack_loss_grad(
        model._stack, batch.handle, _ptr(Xd), _ptr(Ld), _ptr(y), _ptr(w), 1.0 / B, _ptr(model.flat_params.flat),
        _ptr(model.flat_grad), _ptr(model._loss), _ptr(model._arena), model._arena.numel(), cb, None,
        _stream_ptr(DEV)))
    torch.cuda.synchronize()
    nn = len(model.layers)
    assert stages == [nn] + list(range(nn - 1, -1, -1))
    covered = torch.zeros(model.n_parameters(), dtype=torch.int32)
    for s in stages:
        a, b = model._stage_slices[s]
        covered[a:b] += 1
    assert bool((covered == 1).all())


def test_node_list_stack_equals_the_layer_list_stack():
    """A plain SGC_LL stack built through agcn_stack_create_nodes gives what agcn_stack_create gives, bit for bit, with
    the same number of launches per training step and per prediction."""
    from agcn_b200 import _lib
    from agcn_b200.simple_agcn import SimpleAGCNStep, _layer_desc
    B = 256
    X, L, n, batch, Xd, Ld = _inputs(B)
    y, w = _labels(B, 12, "sigmoid_ce")

    class NodeList(SimpleAGCNStep):
        def _create_stack(self, offs):
            nodes = (_lib.StackNode * len(self.layers))()
            for i, l in enumerate(self.layers):
                nodes[i] = _lib.StackNode(_lib.NODE["sgcll"], _layer_desc(l), -1)
            _lib.check(_lib.lib().agcn_stack_create_nodes(nodes, len(self.layers), self.Fm, self.Nt,
                                                          _lib.LOSS[self.loss_kind], offs, ctypes.byref(self._stack)))

    out = []
    for cls in (SimpleAGCNStep, NodeList):
        model = cls(75, (64, 128, 128, 64), 256, 12, 3, B, device=DEV, seed=11)
        model.loss_and_grads(Xd, Ld, batch, y, w)
        model.predict_proba(Xd, Ld, batch)
        torch.cuda.synchronize()
        c0 = _lib.launch_count()
        loss = float(model.loss_and_grads(Xd, Ld, batch, y, w))
        c1 = _lib.launch_count()
        probs, loss_e = model.evaluate(Xd, Ld, batch, y, w)
        c2_ = _lib.launch_count()
        torch.cuda.synchronize()
        out.append((loss, model.flat_grad.detach().clone(), probs, float(loss_e), c1 - c0, c2_ - c1))
    (l0, g0, p0, e0, n0, m0), (l1, g1, p1, e1, n1, m1) = out
    print("launches per step %d / %d, per prediction %d / %d" % (n0, n1, m0, m1))
    assert l0 == l1 and e0 == e1 and torch.equal(g0, g1) and torch.equal(p0, p1)
    assert n0 == n1 and m0 == m1
