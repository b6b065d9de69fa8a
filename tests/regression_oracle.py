"""fp64 reference of the regression head (loss="weighted_l2").  TEST INFRASTRUCTURE ONLY, like
oracle/network_oracle.py, whose DenseMol / GraphGatherMol restatement it follows and whose functions it leaves alone.

  head_values       x [B, T] = tanh(gather(DenseMol(H))) head_W + head_b: one [Fm, 1] fully connected layer per task,
                    no activation (what the regressor predicts).
  weighted_l2       scale * sum_b sum_t (w[b, t] (x[b, t] - y[b, t]))^2 -- DeepChem 1.x MultitaskGraphRegressor's default
                    final_loss='weighted_L2': tf.square(tf.mul(tf.sub(x, t), w)), summed over the batch and the tasks,
                    divided by the batch size.  The weight enters squared.
  weighted_l2_grad  its closed-form gradient d loss / d x = 2 w^2 (x - y) scale.

Parity unpinned, like the other TensorFlow ops of oracle/network_oracle.py: the reference's
models/tf_modules/multitask_regressor.py is restated here, not run.
"""
import torch

from oracle import network_oracle as NO


def head_values(H_list, head_params):
    """H_list: B tensors [n_g, Fh] (the real rows of the last SGC-LL layer's output); head_params: dict dense_W,
    dense_b, head_W [Fm, T], head_b [T].  Returns x [B, T] in the dtype of the inputs."""
    mols = [(h @ head_params["dense_W"] + head_params["dense_b"]).sum(0) for h in H_list]   # DenseMol + gather
    return torch.tanh(torch.stack(mols, 0)) @ head_params["head_W"] + head_params["head_b"]


def weighted_l2(x, targets, weights, scale):
    return ((weights * (x - targets)) ** 2).sum() * scale


def weighted_l2_grad(x, targets, weights, scale):
    return 2.0 * weights * weights * (x - targets) * scale


def simple_agcn_loss(X, L, n_nodes, layer_params, head_params, targets, weights, global_batch, K,
                     laplacian="reference_literal", metric_grad="reference", relu_masks=None):
    """The regressor's counterpart of network_oracle.simple_agcn_loss (same arguments, targets / weights [B, T])."""
    H = NO.simple_agcn_features(X, L, n_nodes, layer_params, K, laplacian, metric_grad, relu_masks)
    return weighted_l2(head_values(H, head_params), targets, weights, 1.0 / global_batch)
