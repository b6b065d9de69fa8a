"""fp64 reference of the per-node classification head (loss="node_softmax_ce").  TEST INFRASTRUCTURE ONLY.

  node_logits     x = H head_W + head_b over every node, the graphs' rows concatenated in packed order
  node_softmax_ce scale * sum_r w_r sum_c y_rc (logsumexp(x_r) - x_rc)
  node_ce_grad    its closed-form gradient w.r.t. x: w_r (softmax_c(x_r) sum_c y_rc - y_rc) scale
  node_agcn_loss  the body of residual_oracle.res_agcn_features (plain SGC_LL stacks are node lists without src, so
                  SimpleAGCNStep and ResAGCNStep share it), then the head and loss above

Restated from the reference's segmentation module, which is not available here: parity unpinned.
"""
import torch

import residual_oracle as RES


def node_logits(H, head_W, head_b):
    """H: list of [n_g, Fh] per graph (or one [R, Fh] tensor) -> x [R, C]."""
    if isinstance(H, (list, tuple)):
        H = torch.cat(list(H), 0)
    return H @ head_W + head_b


def node_softmax_ce(x, targets, weights, scale):
    return ((torch.logsumexp(x, 1) - (x * targets).sum(1)) * weights).sum() * scale


def node_ce_grad(x, targets, weights, scale):
    return weights[:, None] * (torch.softmax(x, 1) * targets.sum(1, keepdim=True) - targets) * scale


def node_agcn_loss(X, L, n_nodes, node_params, srcs, head_params, targets, weights, global_batch, K,
                   laplacian="reference_literal", metric_grad="reference", relu_masks=None):
    H = RES.res_agcn_features(X, L, n_nodes, node_params, srcs, K, laplacian, metric_grad, relu_masks)
    x = node_logits(H, head_params["head_W"], head_params["head_b"])
    return node_softmax_ce(x, targets, weights, 1.0 / global_batch), x
