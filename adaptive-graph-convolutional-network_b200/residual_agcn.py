"""Residual AGCN training step: SGC_LL_Reslap layers chained through their learned Laplacians, in residual blocks
closed by BlockEnd, then the SimpleAGCN head (DenseMol, GraphGatherMol, logits / regression outputs, loss) and Adam.

The reference builds this body with ResidualGraphMolResLap (models/networks/tf_graphs.py:159-223): every Reslap layer
after the first takes the previous Reslap layer's L_all as its L_prev,

    L_all = leaky_alpha(clip(leaky_alpha(clip(res_L)) + L_int + beta L_prev))       (graphconv_reslap.py:91-230)

and BlockEnd adds the block's input through a learned map: act(x_res W + x) (blockend.py:67-86).  In the default
reference_literal mode this chain is where the graph adapts: SGC_LL's own learned Laplacian is the identity there.

Layout, for filters = (f0, f1, ..., fm) and `block`: node 0 is Reslap(n_feat -> f0) with no L_prev; then fm layers in
blocks of `block` Reslap layers, each block closed by BlockEnd(relu) whose x_res is the block's input.  The default
filters=(64, 64, 64, 64, 64), block=2 gives R0, R1, R2, BE(src=R0), R4, R5, BE(src=BE3).  This layout follows the
contracts of the two containers above; ResAGCN.py itself is not available, so parity with its exact layout (depths,
widths, where blocks close) is unpinned.

engine="stack" runs the step as ONE agcn_stack_loss_grad call on a stack of nodes (agcn_stack_create_nodes) and
prediction as one agcn_stack_predict call; engine="autograd" runs the SGC_LL_Reslap and BlockEnd layer classes under
torch.autograd, wired as ResidualGraphMolResLap wires them.  Both give the same numbers bit for bit.  Everything else
(flat buffers, Adam, step / step_graphed, predict_proba / predict / evaluate, the three loss kinds, overlapped
all-reduce buckets) is SimpleAGCNStep's.
"""
import ctypes

from . import _lib
from .layers import BlockEnd, SGC_LL_Reslap
from .layers.blockend import fused_activation
from .simple_agcn import SimpleAGCNStep, _layer_desc


class ResAGCNStep(SimpleAGCNStep):
    def __init__(self, n_feat=75, filters=(64, 64, 64, 64, 64), final_feature_n=256, n_tasks=12, K=3, batch_size=256,
                 block=2, **kwargs):
        """Arguments as SimpleAGCNStep, plus `block`: Reslap layers per residual block.  len(filters) - 1 must be a
        positive multiple of `block`."""
        if block < 1 or len(filters) < 2 or (len(filters) - 1) % block:
            raise ValueError("len(filters) - 1 must be a positive multiple of block (%d filters, block %d)"
                             % (len(filters), block))
        self.block = block
        super(ResAGCNStep, self).__init__(n_feat, filters, final_feature_n, n_tasks, K, batch_size, **kwargs)

    def _build_layers(self, n_feat, filters, batch_size, K, laplacian, metric_grad):
        """self.layers and self.srcs (per node: the Reslap layer whose L_all is its L_prev, or the node whose output
        is a BlockEnd's x_res; -1 for none)."""
        def reslap(fin, fout):
            return SGC_LL_Reslap(fout, fin, batch_size, K=K, activation='relu', laplacian=laplacian,
                                 metric_grad=metric_grad)

        self.layers, self.srcs = [reslap(n_feat, filters[0])], [-1]
        last_reslap, block_in = 0, 0
        for j in range(1, len(filters)):
            self.layers.append(reslap(filters[j - 1], filters[j]))
            self.srcs.append(last_reslap)
            last_reslap = len(self.layers) - 1
            if j % self.block == 0:
                self.layers.append(BlockEnd(len(self.layers), _width(self.layers[block_in]), filters[j],
                                            activation='relu', batch_size=batch_size))
                self.srcs.append(block_in)
                block_in = len(self.layers) - 1

    def nodes(self):
        """The agcn_stack_node array of the body."""
        arr = (_lib.StackNode * len(self.layers))()
        for i, (l, src) in enumerate(zip(self.layers, self.srcs)):
            if isinstance(l, BlockEnd):
                act, host_act = fused_activation(l.activation)
                if host_act is not None:
                    raise ValueError("node %d: a BlockEnd in the stack must be relu or linear (its activation is "
                                     "fused into the product)" % i)
                arr[i] = _lib.StackNode(_lib.NODE["block_end"],
                                        _lib.Desc(l.res_n_features, l.n_features, 0, 0, 0, 0, _lib.ACT[act], 0), src)
            else:
                arr[i] = _lib.StackNode(_lib.NODE["sgcll"], _layer_desc(l), src)
        return arr

    def _create_stack(self, offs):
        _lib.check(_lib.lib().agcn_stack_create_nodes(self.nodes(), len(self.layers), self.Fm, self.Nt,
                                                      _lib.loss_code(self.loss_kind), offs, ctypes.byref(self._stack)))

    def _body(self, x):
        outs, lall = [], {}
        for i, (layer, src) in enumerate(zip(self.layers, self.srcs)):
            if isinstance(layer, BlockEnd):
                out = layer(dict(x, block_outputs=outs[src]))                    # blockend.py:46-65
            elif isinstance(layer, SGC_LL_Reslap):
                out, _, _, lall[i] = layer(dict(x, res_lap=lall[src] if src >= 0 else []))
            else:                                                                   # plain SGC_LL: no L_all
                out, _, _ = layer(x)
            outs.append(out)
            x = dict(x, node_features=out)
        return out

    def loss_and_grads(self, X, Lint, batch, targets, weights):
        if self.engine == "autograd":
            # BlockEnd's weight gradient is accumulated into its flat-buffer view by autograd (the other producers
            # overwrite theirs)
            for l in self.layers:
                if isinstance(l, BlockEnd):
                    l.vars["weight"].grad.zero_()
        return super(ResAGCNStep, self).loss_and_grads(X, Lint, batch, targets, weights)


def _width(layer):
    return layer.n_features if isinstance(layer, BlockEnd) else layer.nb_filter
