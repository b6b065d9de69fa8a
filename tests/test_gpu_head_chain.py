"""The graph head's chain (agcn_head_loss_grad_ex) against float64: hsum -> pre -> tanh -> logits and loss -> dpre ->
dhsum -> dH, and every parameter gradient, at the batch shapes its kernels switch on.

head_fwd_kernel (gather, dense product and tanh) and head_bwd_kernel (split-K partials of dmol, tanh', dhsum and dH)
tile the batch HEAD_GRAPHS = 4 graphs per CTA, so the cases include B = 1, B not a multiple of 4 and 1-, 2- and 3-atom
molecules; above 2^26 multiply-adds dhsum runs on the tensor cores instead ("big").  Nt = 1234 runs dmol split along
K, Nt = 40 / 26 on the tensor cores without a split and Nt = 24 on the CUDA cores.  Every call runs on a non-default
stream with its workspace and outputs filled with NaN bytes first, and only that stream is synchronised before the
outputs are read: each gradient must be complete on the caller's stream, although the parameter gradients run on a
stream of the plan's own.
"""
import ctypes

import numpy as np
import pytest
import torch

DEV = torch.device("cuda:0")
TOL = 1e-4  # max |a - b| / max |b|, as the other fp64 comparisons of the suite


def _sizes(key, rng):
    if key == "tox":
        return rng.integers(1, 60, 1024)
    if key == "tox256":
        return rng.integers(1, 60, 256)
    if key == "one":
        return np.array([23])
    if key == "tiny":
        return np.array([1, 2, 3, 1, 3, 2, 2, 1, 3])
    if key == "tox1023":
        return rng.integers(1, 60, 1023)
    if key == "tox1100":
        return rng.integers(1, 60, 1100)
    if key == "small37":
        return rng.integers(1, 30, 37)
    if key == "modelnet":
        return np.full(32, 1024)
    if key == "sydney":
        return np.exp(rng.uniform(np.log(13), np.log(1024), 128)).astype(np.int64)
    if key == "reg300":
        return rng.integers(1, 60, 300)
    raise KeyError(key)


CASES = [
    # id,        sizes,      Fh,  Fm,  Nt,   loss
    ("C1",       "tox256",   64,  256, 24,   "sigmoid_ce"),   # dmol on the CUDA cores
    ("C2",       "tox",      64,  256, 1234, "sigmoid_ce"),   # dmol split along K
    ("B1",       "one",      64,  256, 1234, "sigmoid_ce"),
    ("tiny",     "tiny",     64,  256, 40,   "sigmoid_ce"),   # 1-3 atoms, B = 9; tensor cores without split
    ("B1023",    "tox1023",  128, 256, 1234, "sigmoid_ce"),
    ("Fm32",     "small37",  40,  32,  24,   "sigmoid_ce"),   # Fh % 32 != 0: the plain row sum
    ("Fm32_128", "small37",  128, 32,  40,   "sigmoid_ce"),
    ("C3",       "modelnet", 64,  256, 40,   "softmax_ce"),
    ("C4",       "sydney",   64,  256, 26,   "softmax_ce"),
    ("L2",       "reg300",   128, 256, 617,  "weighted_l2"),  # split along K
    ("big",      "tox1100",  128, 512, 1234, "sigmoid_ce"),   # B Fh Fm > 2^26: dhsum on the tensor cores
]


def _reference(H, n, p, y, w, scale, loss):
    """float64 head: the loss and d loss / d (H, dense_W, dense_b, head_W, head_b)."""
    H = H.clone().requires_grad_(True)
    p = [t.clone().requires_grad_(True) for t in p]
    dense_W, dense_b, head_W, head_b = p
    graph = torch.repeat_interleave(torch.arange(len(n)), torch.tensor(n))
    hsum = torch.zeros(len(n), H.shape[1], dtype=torch.float64).index_add(0, graph, H)
    mol = torch.tanh(hsum @ dense_W + torch.tensor(n, dtype=torch.float64)[:, None] * dense_b)
    x = mol @ head_W + head_b
    if loss == "sigmoid_ce":
        terms = w * (torch.clamp(x, min=0) - x * y + torch.log1p(torch.exp(-x.abs())))
    elif loss == "softmax_ce":
        terms = w * (torch.logsumexp(x, 1) - (x * y).sum(1))
    else:
        terms = (w * (x - y)) ** 2
    total = terms.sum() * scale
    total.backward()
    return float(total.detach()), [H.grad] + [t.grad for t in p]


def _rel(a, b):
    return float((a.double().cpu() - b).abs().max() / b.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("name,sizes,Fh,Fm,Nt,loss", CASES, ids=[c[0] for c in CASES])
def test_head_chain_matches_fp64(name, sizes, Fh, Fm, Nt, loss):
    import agcn_b200
    from agcn_b200 import _lib
    from agcn_b200.batch import _ptr

    rng = np.random.default_rng(Fh * 7919 + Nt)
    n = np.asarray(_sizes(sizes, rng), np.int32)
    B, R = len(n), int(n.sum())
    H = torch.tensor(np.maximum(rng.standard_normal((R, Fh)), 0) * 0.3)
    p = [torch.tensor(rng.standard_normal(s) * sc) for s, sc in (((Fh, Fm), 0.1 / np.sqrt(Fh / 64)), ((Fm,), 0.05),
                                                                  ((Fm, Nt), 0.1), ((Nt,), 0.1))]
    if loss == "sigmoid_ce":
        y = torch.tensor((rng.random((B, Nt)) < 0.3).astype(np.float64))
        w = torch.tensor(rng.random((B, Nt)) + 0.5)
    elif loss == "softmax_ce":
        y = torch.zeros(B, Nt, dtype=torch.float64)
        y[torch.arange(B), torch.tensor(rng.integers(0, Nt, B))] = 1.0
        w = torch.tensor(rng.random(B) + 0.5)
    else:
        y = torch.tensor(rng.standard_normal((B, Nt)))
        w = torch.tensor((rng.random((B, Nt)) < 0.8).astype(np.float64))
    scale = 1.0 / B
    loss_ref, grads_ref = _reference(H, n, p, y, w, scale, loss)

    stream = torch.cuda.Stream(device=DEV)
    with torch.cuda.stream(stream):
        batch = agcn_b200.GraphBatch(n, int(n.max()), device=DEV)
        lib = _lib.lib()
        nbytes = ctypes.c_size_t()
        _lib.check(lib.agcn_head_workspace_bytes(batch.handle, Fh, Fm, Nt, ctypes.byref(nbytes)))
        work = torch.full((nbytes.value,), 0xFF, dtype=torch.uint8, device=DEV)   # NaN in every float
        Hd, yd, wd = (t.float().to(DEV) for t in (H, y, w))
        pd = [t.float().to(DEV) for t in p]
        nan = float("nan")
        out_loss = torch.full((1,), nan, device=DEV)
        grads = [torch.full_like(t, nan) for t in [Hd] + pd]
        _lib.check(lib.agcn_head_loss_grad_ex(
            batch.handle, _ptr(Hd), _ptr(pd[0]), _ptr(pd[1]), _ptr(pd[2]), _ptr(pd[3]), _ptr(yd), _ptr(wd),
            scale, _lib.LOSS[loss], Fh, Fm, Nt, _ptr(out_loss), *[_ptr(g) for g in grads], _ptr(work), work.numel(),
            ctypes.c_void_p(stream.cuda_stream)))
    stream.synchronize()
    assert abs(float(out_loss) - loss_ref) <= TOL * abs(loss_ref), (float(out_loss), loss_ref)
    for g, r, what in zip(grads, grads_ref, ("dH", "ddense_W", "ddense_b", "dhead_W", "dhead_b")):
        assert torch.isfinite(g).all(), what
        assert _rel(g, r) <= TOL, (what, _rel(g, r))
