"""fp64 reference of the head's class probabilities (predict_proba of the reference's classifiers).  TEST
INFRASTRUCTURE ONLY, like oracle/network_oracle.py, whose DenseMol / GraphGatherMol restatement it follows.

  sigmoid_ce  [B, T, 2]: the softmax over every task's two logits (column 2 t + c of head_W = class c of task t), as
              DeepChem's MultitaskGraphClassifier.predict_proba computes it.
  softmax_ce  [B, C]: the softmax over the class logits (SingletaskGraphClassifier).

Parity unpinned, like the other TensorFlow ops of oracle/network_oracle.py: the reference's classifier sources are
restated here, not run.
"""
import torch


def head_predict(H_list, head_params, loss_kind):
    """H_list: B tensors [n_g, Fh] (the real rows of the last SGC-LL layer's output); head_params: dict dense_W,
    dense_b, head_W, head_b.  Returns the probabilities in the dtype of the inputs (fp64 in the tests)."""
    mols = [(h @ head_params["dense_W"] + head_params["dense_b"]).sum(0) for h in H_list]   # DenseMol + gather
    logits = torch.tanh(torch.stack(mols, 0)) @ head_params["head_W"] + head_params["head_b"]
    if loss_kind == "sigmoid_ce":
        return torch.softmax(logits.reshape(logits.shape[0], -1, 2), -1)
    if loss_kind == "softmax_ce":
        return torch.softmax(logits, -1)
    raise ValueError("unknown loss_kind %r" % (loss_kind,))
