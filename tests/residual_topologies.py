"""Node topologies of the residual stack (agcn_stack_create_nodes) beyond ResAGCNStep's default layout, and a
ResAGCNStep whose body is one of them.  TEST INFRASTRUCTURE ONLY: tests/test_gpu_residual_topologies.py runs them on
the device, tests/test_residual_host.py checks that the stack accepts them and how their parameters are laid out.

Node notation: R = SGC_LL_Reslap, S = plain SGC_LL, BE = BlockEnd; node(src).
"""
N_FEAT = 75

# ("R", Fo, src) / ("S", Fo) / ("BE", src[, "linear"]): a layer's F is the previous node's width (N_FEAT for node 0);
# a BlockEnd's F is the width of H[src] and its Fo the width of H[i-1].
TOPOLOGIES = {
    # a block of one layer; the Reslap chain R1 -> R3 skips over a BlockEnd
    "block1": [("R", 64, -1), ("R", 64, 0), ("BE", 0), ("R", 64, 1), ("BE", 2)],
    # src = i-1: x_res is x, so both contributions to dH[i-1] land in one buffer (the copy branch of the backward)
    "xres_is_x": [("R", 64, -1), ("R", 64, 0), ("BE", 1), ("R", 64, 1), ("BE", 3)],
    # consecutive BlockEnds: H1 is x of the first and x_res of the second
    "be_after_be": [("R", 64, -1), ("R", 64, 0), ("BE", 0), ("BE", 1), ("R", 64, 1)],
    # a BlockEnd at node 1 whose src is the first layer (which has no dX unless paper / full)
    "be_first": [("R", 64, -1), ("BE", 0), ("R", 64, 0), ("BE", 1)],
    # nested blocks: H0 lives until node 5 and H1 until node 4, so prediction needs four activation slots
    "long_range": [("R", 64, -1), ("R", 64, 0), ("R", 64, 1), ("R", 64, 2), ("BE", 1), ("BE", 0)],
    # interleaved L_all chains R0 -> R2 and R1 -> R3: two L_all slots live at once
    "two_chains": [("R", 64, -1), ("R", 64, -1), ("R", 64, 0), ("R", 64, 1), ("BE", 0)],
    # plain layers mixed in; a chain restarting mid-stack (R1) and crossing a BlockEnd and a plain layer (R2 -> R5)
    "mixed_plain": [("S", 64), ("R", 64, -1), ("R", 64, 1), ("BE", 0), ("S", 64), ("R", 64, 2)],
    # F > 128 and F % 4 != 0 (CUDA-core TN and scalar gemm_rows products), F != Fo, a linear BlockEnd feeding the head
    "widths": [("R", 160, -1), ("R", 30, 0), ("BE", 0), ("R", 48, 1), ("BE", 2, "linear")],
}


def widths(spec):
    """Per node (kind, F, Fo, src, activation)."""
    out = []
    for i, node in enumerate(spec):
        if node[0] == "BE":
            src = node[1]
            out.append(("BE", out[src][2], out[i - 1][2], src, node[2] if len(node) > 2 else "relu"))
        else:
            F = N_FEAT if i == 0 else out[i - 1][2]
            out.append((node[0], F, node[1], node[2] if node[0] == "R" else -1, "relu"))
    return out


def topology_model(spec, create_stack=None, **kwargs):
    """A ResAGCNStep whose body is the node list `spec` (TOPOLOGIES); kwargs as ResAGCNStep's.  create_stack(model,
    offsets), if given, sees the flat-buffer offsets the stack is created with."""
    from agcn_b200 import BlockEnd, SGC_LL, SGC_LL_Reslap
    from agcn_b200.residual_agcn import ResAGCNStep

    class TopologyStep(ResAGCNStep):
        def _build_layers(self, n_feat, filters, batch_size, K, laplacian, metric_grad):
            self.layers, self.srcs = [], []
            for i, (kind, F, Fo, src, act) in enumerate(widths(spec)):
                if kind == "BE":
                    layer = BlockEnd(i, F, Fo, activation=act, batch_size=batch_size)
                else:
                    cls = SGC_LL_Reslap if kind == "R" else SGC_LL
                    layer = cls(Fo, F, batch_size, K=K, activation='relu', laplacian=laplacian,
                                metric_grad=metric_grad)
                self.layers.append(layer)
                self.srcs.append(src)

        def _create_stack(self, offs):
            if create_stack is not None:
                create_stack(self, offs)
            super(TopologyStep, self)._create_stack(offs)

    # filters[-1] sizes dense_W: the width of the last node
    filters = tuple(w[2] for w in widths(spec))
    return TopologyStep(N_FEAT, filters, block=1, **kwargs)
