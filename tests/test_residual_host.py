"""The residual stack (agcn_stack_create_nodes, ResAGCNStep) without a GPU: the node constants of the C ABI and their
binding, every rejection of agcn_stack_create_nodes with its message, the default layout accepted, ResAGCNStep's
argument checks and flat-buffer offsets, every topology of the device sweep accepted and laid out, and the residual
oracle's BlockEnd gradient against its closed form."""
import ctypes
import os
import re

import pytest
import torch

import residual_oracle as RES
import residual_topologies as RT
from oracle import sgcll_oracle as O

AGCN_ERR_INVALID = -1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _last_error():
    from agcn_b200 import _lib
    return _lib.lib().agcn_last_error().decode()


def test_node_constants_match_the_header():
    from agcn_b200 import _lib
    with open(os.path.join(ROOT, "include", "agcn_sgcll.h")) as f:
        defines = dict((k, int(v)) for k, v in re.findall(r"#define AGCN_NODE_(\w+) (\d+)", f.read()))
    assert defines == {"SGCLL": 0, "BLOCK_END": 1}
    assert _lib.NODE == {k.lower(): v for k, v in defines.items()}
    assert "agcn_stack_create_nodes" in _lib.EXPORTED_SYMBOLS


def _reslap(F, Fo, src):
    return (0, (F, Fo, 3, 1, 0, 0, 1, 0), src)


def _sgcll(F, Fo, src=-1):
    return (0, (F, Fo, 3, 0, 0, 0, 1, 0), src)


def _block_end(F, Fo, src):
    return (1, (F, Fo, 0, 0, 0, 0, 1, 0), src)


DEFAULT = [_reslap(75, 64, -1), _reslap(64, 64, 0), _reslap(64, 64, 1), _block_end(64, 64, 0), _reslap(64, 64, 2),
           _reslap(64, 64, 4), _block_end(64, 64, 3)]


def _create(spec, offs=None):
    """(return code, last error) of agcn_stack_create_nodes on `spec` [(kind, desc tuple, src)]; offsets default to
    5 distinct ones per node with beta on every Reslap node."""
    from agcn_b200 import _lib
    lib = _lib.lib()
    arr = (_lib.StackNode * len(spec))()
    for i, (kind, d, src) in enumerate(spec):
        arr[i] = _lib.StackNode(kind, _lib.Desc(*d), src)
    if offs is None:
        offs = list(range(5 * len(spec) + 4))
    offs_c = (ctypes.c_int64 * len(offs))(*offs)
    stack = ctypes.c_void_p()
    rc = lib.agcn_stack_create_nodes(arr, len(spec), 256, 24, 0, offs_c, ctypes.byref(stack))
    err = _last_error()
    if stack:
        lib.agcn_stack_destroy(stack)
    assert bool(stack) == (rc == 0)
    return rc, err


def test_create_nodes_accepts_the_default_layout_and_plain_stacks():
    assert _create(DEFAULT)[0] == 0
    assert _create([_sgcll(75, 64), _sgcll(64, 128), _sgcll(128, 64)])[0] == 0
    # a BlockEnd whose x_res is the node right before it, and one fed by a BlockEnd's output: both are expressible
    assert _create([_reslap(75, 64, -1), _block_end(64, 64, 0)])[0] == 0
    assert _create([_reslap(75, 64, -1), _reslap(64, 64, 0), _block_end(64, 64, 0), _block_end(64, 64, 1)])[0] == 0


REJECTIONS = [
    # name, spec, offsets (None: default), message fragment
    ("unknown_kind", [_reslap(75, 64, -1), (2, (64, 64, 0, 0, 0, 0, 1, 0), 0)], None, "node 1: unknown kind"),
    ("unknown_variant", [(0, (75, 64, 3, 5, 0, 0, 1, 0), -1)], None, "node 0: unknown variant"),
    ("block_end_first", [_block_end(75, 75, 0), _reslap(75, 64, -1)], None, "node 0: a BlockEnd cannot be the first"),
    ("block_end_src_later", [_reslap(75, 64, -1), _reslap(64, 64, 0), _block_end(64, 64, 2)], None,
     "node 2: src must be an earlier node"),
    ("block_end_src_negative", [_reslap(75, 64, -1), _block_end(64, 64, -1)], None,
     "node 1: src must be an earlier node"),
    ("reslap_src_later", [_reslap(75, 64, 1), _reslap(64, 64, -1)], None, "node 0: src must be an earlier node"),
    ("reslap_src_not_reslap", [_sgcll(75, 64), _reslap(64, 64, 0)], None, "node 1: a Reslap src must be a Reslap"),
    ("reslap_src_block_end", [_reslap(75, 64, -1), _block_end(64, 64, 0), _reslap(64, 64, 1)], None,
     "node 2: a Reslap src must be a Reslap"),
    ("two_reslaps_same_src", [_reslap(75, 64, -1), _reslap(64, 64, 0), _reslap(64, 64, 0)], None,
     "node 2: two Reslap layers name the same src"),
    ("two_block_ends_same_src", [_reslap(75, 64, -1), _reslap(64, 64, 0), _block_end(64, 64, 0),
                                 _block_end(64, 64, 0)], None, "node 3: two BlockEnds name the same src"),
    ("layer_widths", [_reslap(75, 64, -1), _reslap(32, 64, 0)], None, "node 1: widths do not chain"),
    ("block_end_res_width", [_reslap(75, 64, -1), _reslap(64, 32, 0), _block_end(75, 32, 0)], None,
     "node 2: widths do not chain"),
    ("block_end_out_width", [_reslap(75, 64, -1), _reslap(64, 32, 0), _block_end(64, 64, 0)], None,
     "node 2: widths do not chain"),
    ("missing_beta", [_reslap(75, 64, -1), _reslap(64, 64, 0)], [0, 1, 2, 3, 4, 5, 6, 7, 8, -1, 9, 10, 11, 12],
     "node 1: a Reslap layer needs a beta offset"),
    ("sgcll_with_src", [_reslap(75, 64, -1), _sgcll(64, 64, 0)], None, "node 1: an SGC_LL layer takes no src"),
]


@pytest.mark.parametrize("name,spec,offs,message", REJECTIONS, ids=[r[0] for r in REJECTIONS])
def test_create_nodes_rejects(name, spec, offs, message):
    rc, err = _create(spec, offs)
    assert rc == AGCN_ERR_INVALID
    assert message in err, err


def test_create_nodes_checks_its_arguments():
    from agcn_b200 import _lib
    lib = _lib.lib()
    arr = (_lib.StackNode * 1)(_lib.StackNode(0, _lib.Desc(75, 64, 3, 1, 0, 0, 1, 0), -1))
    offs = (ctypes.c_int64 * 9)(*range(9))
    stack = ctypes.c_void_p()
    assert lib.agcn_stack_create_nodes(arr, 0, 256, 24, 0, offs, ctypes.byref(stack)) == AGCN_ERR_INVALID
    assert lib.agcn_stack_create_nodes(arr, 1, 256, 24, 7, offs, ctypes.byref(stack)) == AGCN_ERR_INVALID
    assert "unknown loss_kind" in _last_error()
    assert not stack


def test_res_agcn_step_layout_and_flat_buffer_offsets():
    from agcn_b200 import BlockEnd, SGC_LL_Reslap, _lib
    from agcn_b200.residual_agcn import ResAGCNStep
    class Probe(ResAGCNStep):
        def _create_stack(self, offs):
            self.offs = list(offs)
            super(Probe, self)._create_stack(offs)

    model = Probe(device="cpu", batch_size=8)
    kinds = ["R" if isinstance(l, SGC_LL_Reslap) else "BE" for l in model.layers]
    assert kinds == ["R", "R", "R", "BE", "R", "R", "BE"]
    assert model.srcs == [-1, 0, 1, 0, 2, 4, 3]
    nodes = model.nodes()
    assert [nodes[i].kind for i in range(7)] == [0, 0, 0, 1, 0, 0, 1]
    assert [(nodes[i].desc.F, nodes[i].desc.Fo) for i in range(7)] == [(75, 64)] + [(64, 64)] * 6
    assert all(nodes[i].desc.variant == _lib.VARIANT["SGC_LL_Reslap"] for i in (0, 1, 2, 4, 5))
    # the stages of the flat buffer: node after node (weight, bias, M_L, alpha, beta / BlockEnd weight), then the head
    # and the offsets agcn_stack_create_nodes receives: 5 per node, -1 where a node has no such tensor
    off = 0
    base = model.flat_params.flat.data_ptr()
    for i, (l, (a, b)) in enumerate(zip(model.layers, model._stage_slices)):
        assert a == off
        for name, v in l.vars.items():
            assert v.data_ptr() == base + 4 * off
            off += v.numel()
        assert b == off
        want = [(l.vars[k].data_ptr() - base) // 4 if k in l.vars else -1
                for k in ("weight", "bias", "M_L", "alpha", "beta")]
        assert model.offs[5 * i:5 * i + 5] == want
        if isinstance(l, BlockEnd):
            assert list(l.vars) == ["weight"] and tuple(l.vars["weight"].shape) == (64, 64)
        else:
            assert list(l.vars) == ["weight", "bias", "M_L", "alpha", "beta"]
    assert model.offs[35:] == [(getattr(model, k).data_ptr() - base) // 4
                               for k in ("dense_W", "dense_b", "head_W", "head_b")]
    assert model._stage_slices[-1] == (off, model.n_parameters())
    assert model.n_parameters() == off + 64 * 256 + 256 + 256 * 24 + 24
    # a regressor and a softmax head on the same body
    assert ResAGCNStep(device="cpu", loss="weighted_l2", n_tasks=3).Nt == 3
    assert ResAGCNStep(device="cpu", loss="softmax_ce", n_tasks=10).Nt == 10


def test_res_agcn_step_checks_its_arguments():
    from agcn_b200.residual_agcn import ResAGCNStep
    for filters, block in (((64, 64, 64, 64), 2), ((64,), 1), ((64, 64, 64), 0)):
        with pytest.raises(ValueError, match="multiple of block"):
            ResAGCNStep(filters=filters, block=block, device="cpu")
    with pytest.raises(ValueError):
        ResAGCNStep(device="cpu", engine="eager")
    m = ResAGCNStep(filters=(32, 48, 48, 16), block=3, device="cpu")
    assert m.srcs == [-1, 0, 1, 2, 0] and m.layers[-1].res_n_features == 32 and m.layers[-1].n_features == 16


def test_simple_agcn_parameters_are_unchanged_by_the_split_constructor():
    """SimpleAGCNStep's parameters come from the same RNG draws in the same order as before the body was made
    overridable: the first layer's weight is the first glorot draw after manual_seed(seed)."""
    from agcn_b200.simple_agcn import SimpleAGCNStep
    m = SimpleAGCNStep(75, (64, 128, 128, 64), 256, 12, 3, 8, device="cpu", seed=123)
    torch.manual_seed(123)
    lim = (6.0 / (75 * 3 + 64)) ** 0.5
    w = (torch.rand(75 * 3, 64) * 2 - 1) * lim
    assert torch.equal(m.layers[0].vars["weight"].detach(), w)
    assert [list(l.vars) for l in m.layers] == [["weight", "bias", "M_L", "alpha"]] * 4


def test_oracle_block_end_gradient_matches_its_closed_form():
    """R0, R1, BE(src=R0): H = relu(H0 W + H1).  With loss = sum(H * C): dW = sum_g H0_g^T (C_g * [H_g > 0])."""
    g = torch.Generator().manual_seed(4)
    sizes = [5, 9, 3]
    B, Nmax, F, Fo, K = len(sizes), 9, 8, 6, 3
    X = torch.zeros(B, Nmax, F, dtype=torch.float64)
    L = torch.zeros(B, Nmax, Nmax, dtype=torch.float64)
    for b, n in enumerate(sizes):
        X[b, :n] = torch.randn(n, F, generator=g, dtype=torch.float64)
        a = torch.rand(n, n, generator=g, dtype=torch.float64)
        L[b, :n, :n] = (a + a.T) * 0.2
    p0 = O.make_params(F, Fo, K, "SGC_LL_Reslap", seed=1, dtype=torch.float64)
    p1 = O.make_params(Fo, Fo, K, "SGC_LL_Reslap", seed=2, dtype=torch.float64)
    W = (torch.randn(Fo, Fo, generator=g, dtype=torch.float64) * 0.5).requires_grad_(True)
    for p in (p0, p1):
        p["beta"].requires_grad_(True)
    C = [torch.randn(n, Fo, generator=g, dtype=torch.float64) for n in sizes]
    H = RES.res_agcn_features(X, L, sizes, [p0, p1, {"weight": W}], [-1, 0, 0], K, "paper", "reference")
    loss = sum((h * c).sum() for h, c in zip(H, C))
    loss.backward()
    closed = torch.zeros(Fo, Fo, dtype=torch.float64)
    for b, n in enumerate(sizes):
        y0, _, _, l0 = O.sgc_ll_graph(X[b, :n], L[b, :n, :n], p0, K, "SGC_LL_Reslap", "paper", "reference")
        h0 = torch.relu(y0)
        y1, _, _, _ = O.sgc_ll_graph(h0, L[b, :n, :n], p1, K, "SGC_LL_Reslap", "paper", "reference", L_prev=l0)
        h = torch.relu(h0 @ W + torch.relu(y1))
        closed += h0.detach().T @ (C[b] * (h > 0).double())
    assert torch.allclose(W.grad, closed, rtol=1e-12, atol=1e-12)
    assert float(W.grad.abs().max()) > 0
    # the second layer's beta weighs the first layer's L_all (its L_prev)
    assert p1["beta"].grad is not None and float(p1["beta"].grad.abs()) > 0


@pytest.mark.parametrize("name", sorted(RT.TOPOLOGIES))
def test_topology_sweep_is_accepted_and_laid_out(name):
    """Every topology of tests/test_gpu_residual_topologies.py passes agcn_stack_create_nodes' checks, and the model
    built on it hands the stack 5 offsets per node (beta only on Reslap nodes, -1 where a node has no such tensor)
    plus the 4 head tensors, in the order of the flat buffers."""
    from agcn_b200 import BlockEnd, SGC_LL_Reslap, _lib
    spec = RT.widths(RT.TOPOLOGIES[name])
    kind = {"R": 0, "S": 0, "BE": 1}
    variant = {"R": _lib.VARIANT["SGC_LL_Reslap"], "S": _lib.VARIANT["SGC_LL"], "BE": 0}
    assert _create([(kind[k], (F, Fo, 3 if k != "BE" else 0, variant[k], 0, 0, _lib.ACT[act], 0), src)
                    for k, F, Fo, src, act in spec])[0] == 0

    got = {}

    def probe(model, offs):
        got["offs"] = list(offs)

    model = RT.topology_model(RT.TOPOLOGIES[name], batch_size=8, device="cpu", create_stack=probe)
    assert model.srcs == [s[3] for s in spec]
    nodes = model.nodes()
    base = model.flat_params.flat.data_ptr()
    for i, (l, (k, F, Fo, src, act)) in enumerate(zip(model.layers, spec)):
        assert (nodes[i].kind, nodes[i].desc.F, nodes[i].desc.Fo, nodes[i].src) == (kind[k], F, Fo, src)
        assert nodes[i].desc.activation == _lib.ACT[act]
        assert isinstance(l, BlockEnd) == (k == "BE") and isinstance(l, SGC_LL_Reslap) == (k == "R")
        want = [(l.vars[t].data_ptr() - base) // 4 if t in l.vars else -1
                for t in ("weight", "bias", "M_L", "alpha", "beta")]
        assert got["offs"][5 * i:5 * i + 5] == want
        assert (want[4] >= 0) == (k == "R")
        assert (want[1] >= 0) == (k != "BE")
    n = len(spec)
    assert len(got["offs"]) == 5 * n + 4
    assert got["offs"][5 * n:] == [(getattr(model, t).data_ptr() - base) // 4
                                   for t in ("dense_W", "dense_b", "head_W", "head_b")]
    assert tuple(model.dense_W.shape) == (spec[-1][2], 256)


def test_block_end_activation_reaches_the_stack():
    """A BlockEnd node carries its layer's activation (a linear BlockEnd trains linear in the stack, as under autograd);
    one the product cannot fuse is refused."""
    from agcn_b200 import _lib
    spec = [("R", 64, -1), ("R", 64, 0), ("BE", 0, "linear")]
    model = RT.topology_model(spec, batch_size=8, device="cpu")
    assert [model.nodes()[i].desc.activation for i in range(3)] == [_lib.ACT["relu"]] * 2 + [_lib.ACT["linear"]]
    with pytest.raises(ValueError, match="node 2: a BlockEnd in the stack must be relu or linear"):
        RT.topology_model([("R", 64, -1), ("R", 64, 0), ("BE", 0, "tanh")], batch_size=8, device="cpu")
