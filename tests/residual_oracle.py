"""fp64 reference of the residual AGCN body (agcn_b200.residual_agcn.ResAGCNStep).  TEST INFRASTRUCTURE ONLY, like
oracle/network_oracle.py, whose functions it composes and leaves alone:

  res_agcn_features  per graph, node after node: an SGC_LL_Reslap layer is O.sgc_ll_graph(..., "SGC_LL_Reslap",
                     L_prev = the L_all of its src node, or None) followed by relu; a plain SGC_LL layer (no "beta")
                     is O.sgc_ll_graph(..., "SGC_LL", ...) followed by relu and produces no L_all; a BlockEnd node is
                     NO.block_end(H[i-1], H[src], W) = act(H[src] W + H[i-1]), act = relu unless `acts` says
                     "linear" for that node.
  res_agcn_loss      the same, then the head and loss of the given kind (sigmoid CE as NO.head_loss, softmax CE as
                     tests/test_gpu_network.py states it, weighted L2 as tests/regression_oracle.py).

relu_masks (optional): per node a bool tensor [R, Fo] over the packed rows saying which outputs the implementation under
test found positive, for every relu node (SGC_LL and SGC_LL_Reslap layers, relu BlockEnds; a linear BlockEnd's entry
is ignored).  As in NO.simple_agcn_features: a pre-activation within rounding error of 0 can land on either side in two
correct implementations, so with the masks given relu(y) is evaluated as y * mask and both sides differentiate the same
piecewise-linear branch.

Parity unpinned, like the other TensorFlow containers of oracle/network_oracle.py.
"""
import torch

import regression_oracle as RO
from oracle import network_oracle as NO
from oracle import sgcll_oracle as O


def res_agcn_features(X, L, n_nodes, node_params, srcs, K, laplacian="reference_literal", metric_grad="reference",
                      relu_masks=None, acts=None):
    """X [B,Nmax,F], L [B,Nmax,Nmax], n_nodes [B]; node_params: per node the dict of its parameters (a BlockEnd has
    only "weight", a plain SGC_LL layer no "beta"); srcs: per node the src of agcn_stack_node; acts: per node "relu" or
    "linear" (None: relu everywhere; only a BlockEnd may be linear).  Returns the B [n_g, Fo] outputs of the last
    node."""
    acts = ["relu"] * len(node_params) if acts is None else acts
    H, row = [], 0
    skip = laplacian == "reference_literal"
    for g in range(X.shape[0]):
        n = int(n_nodes[g])
        x, Lg = X[g, :n], L[g, :n, :n]
        outs, lall = [], {}
        for i, (p, src) in enumerate(zip(node_params, srcs)):
            if acts[i] == "linear":
                act = _identity
            elif relu_masks is None:
                act = torch.relu
            else:
                mask = relu_masks[i][row:row + n]
                act = lambda y, m=mask: y * m.to(y.dtype)       # noqa: E731
            if "M_L" not in p:                                  # BlockEnd, blockend.py:67-86
                x = NO.block_end(x, outs[src], p["weight"], act)
            elif "beta" in p:                                   # SGC_LL_Reslap, graphconv_reslap.py:91-230
                y, _, _, lall[i] = O.sgc_ll_graph(x, Lg, p, K, "SGC_LL_Reslap", laplacian, metric_grad,
                                                  L_prev=lall[src] if src >= 0 else None, compute_similarity=not skip)
                x = act(y)
            else:                                               # SGC_LL, graphconv.py:85-125
                y, _, _, _ = O.sgc_ll_graph(x, Lg, p, K, "SGC_LL", laplacian, metric_grad, compute_similarity=not skip)
                x = act(y)
            outs.append(x)
        H.append(x)
        row += n
    return H


def _identity(y):
    return y


def head_loss(H, head_params, targets, weights, scale, loss_kind):
    if loss_kind == "sigmoid_ce":
        return NO.head_loss(H, head_params["dense_W"], head_params["dense_b"], head_params["head_W"],
                            head_params["head_b"], targets, weights, scale)
    logits = RO.head_values(H, head_params)
    if loss_kind == "weighted_l2":
        return RO.weighted_l2(logits, targets, weights, scale)
    if loss_kind == "softmax_ce":
        return ((torch.logsumexp(logits, 1) - (logits * targets).sum(1)) * weights).sum() * scale
    raise ValueError("unknown loss_kind %r" % (loss_kind,))


def res_agcn_loss(X, L, n_nodes, node_params, srcs, head_params, targets, weights, global_batch, K, loss_kind,
                  laplacian="reference_literal", metric_grad="reference", relu_masks=None, acts=None):
    H = res_agcn_features(X, L, n_nodes, node_params, srcs, K, laplacian, metric_grad, relu_masks, acts)
    return head_loss(H, head_params, targets, weights, 1.0 / global_batch, loss_kind)
