"""torch.autograd bridge to the C ABI: the SGC-LL layer on packed tensors."""
import ctypes

import torch

from . import _lib
from .batch import GraphBatch, _ptr, _stream_ptr


class _Workspace(object):
    """Grow-only scratch buffer per (device, stream) (the `work` area of agcn_sgcll_forward/backward): calls on
    one stream are ordered, so they can share it; calls on different streams must not."""
    _bufs = {}

    @classmethod
    def get(cls, device, nbytes):
        key = (device, torch.cuda.current_stream(device).cuda_stream)
        buf = cls._bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(int(nbytes * 1.25) + 1024, dtype=torch.uint8, device=device)
            cls._bufs[key] = buf
        return buf


def make_desc(F, Fo, K, variant, laplacian, metric_grad, activation, flags):
    return _lib.Desc(F, Fo, K, _lib.VARIANT[variant], _lib.LAPLACIAN[laplacian], _lib.METRIC_GRAD[metric_grad],
                     _lib.ACT[activation], flags)


class _SGCLLFunction(torch.autograd.Function):
    """Forward/backward of SGC_LL.specgraph_LL (graphconv.py:127-252) / specgraph_LL_reslap
    (graphconv_reslap.py:91-230) for one packed batch."""

    @staticmethod
    def forward(ctx, X, Lint, Lprev, M_L, weight, bias, alpha, beta, batch, cfg):
        F, Fo, K = cfg["F"], cfg["Fo"], cfg["K"]
        flags = _lib.SAVE_FOR_BACKWARD
        want_resL, want_resW = cfg.get("want_resL", False), cfg.get("want_resW", False)
        reslap = cfg["variant"] == "SGC_LL_Reslap"
        if want_resL:
            flags |= _lib.OUT_RES_L
        if want_resW:
            flags |= _lib.OUT_RES_W
        if reslap:
            flags |= _lib.OUT_L_ALL
        desc = make_desc(F, Fo, K, cfg["variant"], cfg["laplacian"], cfg["metric_grad"], cfg["activation"], flags)
        X = X.contiguous()
        Lint = Lint.contiguous()
        if Lprev is not None:
            Lprev = Lprev.contiguous()
        assert X.shape == (batch.total_nodes, F) and X.dtype == torch.float32 and X.is_cuda
        assert Lint.numel() == batch.total_lap
        dev = X.device
        saved_b, work_b = ctypes.c_size_t(), ctypes.c_size_t()
        _lib.check(_lib.lib().agcn_sgcll_workspace_bytes(ctypes.byref(desc), batch.handle, ctypes.byref(saved_b),
                                                         ctypes.byref(work_b)))
        saved = torch.empty(saved_b.value, dtype=torch.uint8, device=dev)
        work = _Workspace.get(dev, work_b.value)
        Y = torch.empty(batch.total_nodes, Fo, device=dev, dtype=torch.float32)
        resL = torch.empty(batch.total_lap, device=dev, dtype=torch.float32) if want_resL else None
        resW = torch.empty(batch.total_lap, device=dev, dtype=torch.float32) if want_resW else None
        Lall = torch.empty(batch.total_lap, device=dev, dtype=torch.float32) if reslap else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().agcn_sgcll_forward(
                ctypes.byref(desc), batch.handle, _ptr(X), _ptr(Lint), _ptr(Lprev), _ptr(M_L), _ptr(weight), _ptr(bias),
                _ptr(alpha), _ptr(beta), _ptr(Y), _ptr(resL), _ptr(resW), _ptr(Lall), _ptr(saved), _ptr(work),
                work.numel(), _stream_ptr(dev)))
        ctx.batch, ctx.cfg, ctx.desc = batch, cfg, desc
        # parameters registered with FlatGradBuffer(direct=...): backward writes their gradients in place
        ctx.grad_out = [getattr(t, "_agcn_grad_out", None) if t is not None else None
                        for t in (M_L, weight, bias, alpha, beta)]
        ctx.set_materialize_grads(False)
        ctx.has_prev = Lprev is not None
        ctx.has_beta = beta is not None
        ctx.save_for_backward(X, Lint, Lprev, M_L, weight, alpha, beta, Y, saved)
        outs = [Y, resL, resW, Lall]
        nondiff = [t for t in (resL, resW) if t is not None]
        if nondiff:
            ctx.mark_non_differentiable(*nondiff)
        return tuple(outs)

    @staticmethod
    def backward(ctx, dY, _dresL, _dresW, dLall):
        X, Lint, Lprev, M_L, weight, alpha, beta, Y, saved = ctx.saved_tensors
        batch, cfg, desc = ctx.batch, ctx.cfg, ctx.desc
        F, Fo, K = cfg["F"], cfg["Fo"], cfg["K"]
        dev = X.device
        if dY is None:
            dY = torch.zeros_like(Y)
        dY = dY.contiguous()
        if dLall is not None:
            dLall = dLall.contiguous()
        work_b = ctypes.c_size_t()
        _lib.check(_lib.lib().agcn_sgcll_workspace_bytes(ctypes.byref(desc), batch.handle, None, ctypes.byref(work_b)))
        work = _Workspace.get(dev, work_b.value)
        need_dX = ctx.needs_input_grad[0] or cfg["metric_grad"] == "full"
        dX = torch.empty_like(X) if need_dX else None
        gM, gW, gb, ga, gbeta = ctx.grad_out
        dM = gM if gM is not None else torch.empty_like(M_L)
        dW = gW if gW is not None else torch.empty_like(weight)
        db = gb if gb is not None else torch.empty(Fo, device=dev, dtype=torch.float32)
        dalpha = ga if ga is not None else torch.empty(1, device=dev, dtype=torch.float32)
        dbeta = None
        if ctx.has_beta:
            dbeta = gbeta if gbeta is not None else torch.zeros(1, device=dev, dtype=torch.float32)
        dLprev = torch.empty_like(Lprev) if ctx.has_prev else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().agcn_sgcll_backward(
                ctypes.byref(desc), batch.handle, _ptr(X), _ptr(Lint), _ptr(Lprev), _ptr(M_L), _ptr(weight), _ptr(alpha),
                _ptr(beta), _ptr(Y), _ptr(dY), _ptr(dLall), _ptr(saved), _ptr(dX), _ptr(dM), _ptr(dW), _ptr(db),
                _ptr(dalpha), _ptr(dbeta), _ptr(dLprev), _ptr(work), work.numel(), _stream_ptr(dev)))
        # gradients written in place are not returned (autograd would add them to themselves)
        return (dX, None, dLprev, None if gM is not None else dM, None if gW is not None else dW,
                None if gb is not None else db, None if ga is not None else dalpha,
                None if gbeta is not None else dbeta, None, None)


def sgc_ll_packed(X, Lint, Lprev, params, batch, cfg):
    """X [R,F], Lint packed, Lprev packed or None -> (Y [R,Fo], resL, resW, Lall) packed."""
    return _SGCLLFunction.apply(X, Lint, Lprev, params["M_L"], params["weight"], params["bias"], params["alpha"],
                                params.get("beta"), batch, cfg)


class _HeadLossFunction(torch.autograd.Function):
    """DenseMol + GraphGatherMol(tanh) + multitask logits + weighted sigmoid cross-entropy * scale
    (dense_layer.py:33-50, graphgather.py:50-78, model_operatos.py:792-864, multitask_classifier.py:41-44,187-209),
    or the softmax / weighted-L2 heads (loss_kind) -> scalar loss.  The C call computes the loss AND every gradient; backward hands them out (scaled by the
    incoming gradient unless `unit_grad` says the loss is differentiated directly)."""

    @staticmethod
    def forward(ctx, H, dense_W, dense_b, head_W, head_b, targets, weights, batch, scale, unit_grad, loss_kind):
        H = H.contiguous()
        R, Fh = H.shape
        Fm, Nt = head_W.shape
        dev = H.device
        assert dense_W.shape == (Fh, Fm) and targets.shape == (batch.batch_size, Nt) and R == batch.total_nodes
        assert weights.numel() == (batch.batch_size if loss_kind == "softmax_ce" else batch.batch_size * Nt)
        nbytes = ctypes.c_size_t()
        _lib.check(_lib.lib().agcn_head_workspace_bytes(batch.handle, Fh, Fm, Nt, ctypes.byref(nbytes)))
        work = _Workspace.get(dev, nbytes.value)
        outs = [getattr(t, "_agcn_grad_out", None) for t in (dense_W, dense_b, head_W, head_b)]
        grads = [o if o is not None else torch.empty_like(t) for o, t in zip(outs, (dense_W, dense_b, head_W, head_b))]
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        dH = torch.empty_like(H)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().agcn_head_loss_grad_ex(
                batch.handle, _ptr(H), _ptr(dense_W), _ptr(dense_b), _ptr(head_W), _ptr(head_b),
                _ptr(targets.contiguous()), _ptr(weights.contiguous()), float(scale), _lib.LOSS[loss_kind], Fh, Fm, Nt,
                _ptr(loss), _ptr(dH),
                _ptr(grads[0]), _ptr(grads[1]), _ptr(grads[2]), _ptr(grads[3]), _ptr(work), work.numel(),
                _stream_ptr(dev)))
        ctx.unit_grad = unit_grad
        ctx.in_place = [o is not None for o in outs]
        ctx.save_for_backward(dH, *grads)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        dH, *grads = ctx.saved_tensors
        if not ctx.unit_grad:
            dH = dH * g
            grads = [t if ip else t * g for t, ip in zip(grads, ctx.in_place)]
        # gradients already written into the flat gradient buffer are not returned
        out = [None if ip else t for t, ip in zip(grads, ctx.in_place)]
        return (dH, out[0], out[1], out[2], out[3], None, None, None, None, None, None)


def head_loss(H, dense_W, dense_b, head_W, head_b, targets, weights, batch, scale, unit_grad=False,
              loss_kind="sigmoid_ce"):
    """Scalar loss of the SimpleAGCN head on the packed output of the last SGC-LL layer.
    loss_kind "sigmoid_ce": multitask two-class heads, weights [B, Nt]; "softmax_ce": one n_classes head,
    weights [B]; "weighted_l2": n_tasks regression outputs (Nt = n_tasks), targets / weights [B, Nt] float,
    loss = scale * sum (w (x - y))^2.  unit_grad=True: the caller differentiates this loss directly (d loss / d loss = 1), which skips
    the rescaling kernels; parameters registered with FlatGradBuffer(direct=...) require it."""
    return _HeadLossFunction.apply(H, dense_W, dense_b, head_W, head_b, targets, weights, batch, scale, unit_grad,
                                   loss_kind)


def head_predict(H, dense_W, dense_b, head_W, head_b, batch, loss_kind, targets=None, weights=None, scale=None):
    """Class probabilities of the SimpleAGCN head on the packed output of the last SGC-LL layer (agcn_head_predict),
    with no autograd node.  Returns (probs [B, Nt], loss or None).
    loss_kind "sigmoid_ce": probs[b, 2t+c] = softmax over task t's two logits; "softmax_ce": softmax over the Nt
    class logits; "weighted_l2": the regression values x [B, Nt] themselves, not probabilities.  With targets and
    weights (laid out as for head_loss) the loss is also computed: the same weighted loss x scale as head_loss, bit for
    bit; scale defaults to 1 / batch size."""
    if (targets is None) != (weights is None):
        raise ValueError("head_predict: pass both targets and weights, or neither")
    H = H.detach().contiguous()
    R, Fh = H.shape
    Fm, Nt = head_W.shape
    B = batch.batch_size
    dev = H.device
    assert dense_W.shape == (Fh, Fm) and R == batch.total_nodes
    loss = None
    if targets is not None:
        targets, weights = targets.detach().contiguous(), weights.detach().contiguous()
        assert targets.shape == (B, Nt)
        assert weights.numel() == (B if loss_kind == "softmax_ce" else B * Nt)
        scale = 1.0 / B if scale is None else scale
        loss = torch.empty(1, device=dev, dtype=torch.float32)
    nbytes = ctypes.c_size_t()
    _lib.check(_lib.lib().agcn_head_predict_workspace_bytes(batch.handle, Fh, Fm, Nt, ctypes.byref(nbytes)))
    work = _Workspace.get(dev, nbytes.value)
    probs = torch.empty(B, Nt, device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().agcn_head_predict(
            batch.handle, _ptr(H), _ptr(dense_W.detach()), _ptr(dense_b.detach()), _ptr(head_W.detach()),
            _ptr(head_b.detach()), _ptr(targets), _ptr(weights), float(scale or 0.0), _lib.LOSS[loss_kind], Fh, Fm, Nt,
            _ptr(probs), _ptr(loss), _ptr(work), work.numel(), _stream_ptr(dev)))
    return probs, (loss.reshape(()) if loss is not None else None)


class _NodeHeadLossFunction(torch.autograd.Function):
    """Per-node classification head (agcn_node_head_loss_grad): x = H head_W + head_b for every packed row, softmax
    cross-entropy weighted per node * scale -> scalar loss.  The C call computes the loss AND every gradient; backward
    hands them out as _HeadLossFunction does."""

    @staticmethod
    def forward(ctx, H, head_W, head_b, targets, weights, batch, scale, unit_grad):
        H = H.contiguous()
        R, Fh = H.shape
        C = head_W.shape[1]
        dev = H.device
        assert head_W.shape == (Fh, C) and R == batch.total_nodes
        assert targets.shape == (R, C) and weights.numel() == R
        nbytes = ctypes.c_size_t()
        _lib.check(_lib.lib().agcn_node_head_workspace_bytes(batch.handle, Fh, C, ctypes.byref(nbytes)))
        work = _Workspace.get(dev, nbytes.value)
        outs = [getattr(t, "_agcn_grad_out", None) for t in (head_W, head_b)]
        grads = [o if o is not None else torch.empty_like(t) for o, t in zip(outs, (head_W, head_b))]
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        dH = torch.empty_like(H)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().agcn_node_head_loss_grad(
                batch.handle, _ptr(H), _ptr(head_W), _ptr(head_b), _ptr(targets.contiguous()),
                _ptr(weights.contiguous()), float(scale), Fh, C, _ptr(loss), _ptr(dH), _ptr(grads[0]), _ptr(grads[1]),
                _ptr(work), work.numel(), _stream_ptr(dev)))
        ctx.unit_grad = unit_grad
        ctx.in_place = [o is not None for o in outs]
        ctx.save_for_backward(dH, *grads)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        dH, *grads = ctx.saved_tensors
        if not ctx.unit_grad:
            dH = dH * g
            grads = [t if ip else t * g for t, ip in zip(grads, ctx.in_place)]
        out = [None if ip else t for t, ip in zip(grads, ctx.in_place)]
        return (dH, out[0], out[1], None, None, None, None, None)


def node_head_loss(H, head_W, head_b, targets, weights, batch, scale, unit_grad=False):
    """Scalar loss of the per-node head on the packed output of the last node: H [R, Fh], head_W [Fh, C], head_b [C],
    targets [R, C] one-hot float, weights [R] (0 masks a node); loss = scale * sum_r w_r (logsumexp(x_r) - <y_r, x_r>).
    unit_grad as for head_loss."""
    return _NodeHeadLossFunction.apply(H, head_W, head_b, targets, weights, batch, scale, unit_grad)


def node_head_predict(H, head_W, head_b, batch, targets=None, weights=None, scale=None):
    """Per-node class probabilities (agcn_node_head_predict), no autograd node: (probs [R, C], loss or None).  With
    targets [R, C] and weights [R] the loss is also computed, bit for bit the loss of node_head_loss; scale defaults to
    1 / batch size."""
    if (targets is None) != (weights is None):
        raise ValueError("node_head_predict: pass both targets and weights, or neither")
    H = H.detach().contiguous()
    R, Fh = H.shape
    C = head_W.shape[1]
    dev = H.device
    assert head_W.shape == (Fh, C) and R == batch.total_nodes
    loss = None
    if targets is not None:
        targets, weights = targets.detach().contiguous(), weights.detach().contiguous()
        assert targets.shape == (R, C) and weights.numel() == R
        scale = 1.0 / batch.batch_size if scale is None else scale
        loss = torch.empty(1, device=dev, dtype=torch.float32)
    nbytes = ctypes.c_size_t()
    _lib.check(_lib.lib().agcn_node_head_predict_workspace_bytes(batch.handle, Fh, C, ctypes.byref(nbytes)))
    work = _Workspace.get(dev, nbytes.value)
    probs = torch.empty(R, C, device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().agcn_node_head_predict(
            batch.handle, _ptr(H), _ptr(head_W.detach()), _ptr(head_b.detach()), _ptr(targets), _ptr(weights),
            float(scale or 0.0), Fh, C, _ptr(probs), _ptr(loss), _ptr(work), work.numel(), _stream_ptr(dev)))
    return probs, (loss.reshape(()) if loss is not None else None)


class _UnpackNodes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, packed, batch):
        ctx.batch = batch
        return batch.unpack_nodes(packed)

    @staticmethod
    def backward(ctx, g):
        return ctx.batch.pack_nodes(g), None


class _PackNodes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, padded, batch):
        ctx.batch = batch
        return batch.pack_nodes(padded)

    @staticmethod
    def backward(ctx, g):
        return ctx.batch.unpack_nodes(g), None


def unpack_nodes(packed, batch):
    return _UnpackNodes.apply(packed, batch)


def pack_nodes(padded, batch):
    if not padded.is_cuda:
        # pinned host input (zero-copy read by the pack kernel): an input placeholder, never differentiated --
        # routing it through autograd would hand a CUDA gradient to a CPU tensor
        return batch.pack_nodes(padded)
    return _PackNodes.apply(padded, batch)


class _NodeLinear(torch.autograd.Function):
    """C = act(scale * A W + bias + add) over the packed rows (agcn_node_gemm): the per-graph matmuls of BlockEnd
    (blockend.py:67-86), DenseBlockEnd (densenet_block.py:98-131), MLP (MLP.py:69-83) for the whole batch at once."""

    @staticmethod
    def forward(ctx, A, W, bias, scale, add, act):
        A = A.contiguous()
        W = W.contiguous()
        M, Kd = A.shape
        N = W.shape[1]
        assert W.shape[0] == Kd and A.is_cuda and A.dtype == torch.float32
        dev = A.device
        lib = _lib.lib()
        C = torch.empty(M, N, device=dev, dtype=torch.float32)
        if add is not None:
            C.copy_(add)
        scratch = _Workspace.get(dev, lib.agcn_node_gemm_scratch_bytes(max(N, Kd), max(N, Kd)))
        with torch.cuda.device(dev):
            _lib.check(lib.agcn_node_gemm(_ptr(A), Kd, _ptr(W), N, 0, _ptr(C), N, M, N, Kd, _ptr(bias), _ptr(scale),
                                          1 if add is not None else 0, _lib.ACT[act], _ptr(scratch), _stream_ptr(dev)))
        ctx.act = act
        ctx.has = (bias is not None, scale is not None, add is not None)
        ctx.save_for_backward(A, W, scale, C)
        return C

    @staticmethod
    def backward(ctx, dC):
        A, W, scale, C = ctx.saved_tensors
        has_bias, has_scale, has_add = ctx.has
        dev = A.device
        lib = _lib.lib()
        M, Kd = A.shape
        N = W.shape[1]
        dpre = (dC * (C > 0)) if ctx.act == "relu" else dC
        dpre = dpre.contiguous()
        dA = dW = dbias = dscale = None
        scratch = _Workspace.get(dev, lib.agcn_node_gemm_scratch_bytes(max(N, Kd), max(N, Kd)))
        with torch.cuda.device(dev):
            if ctx.needs_input_grad[0]:
                dA = torch.empty_like(A)          # dA = scale * dpre W^T
                _lib.check(lib.agcn_node_gemm(_ptr(dpre), N, _ptr(W), N, 1, _ptr(dA), Kd, M, Kd, N, None, _ptr(scale), 0,
                                              _lib.ACT["linear"], _ptr(scratch), _stream_ptr(dev)))
            if ctx.needs_input_grad[1] or (has_scale and ctx.needs_input_grad[3]):
                dWu = torch.empty_like(W)         # A^T dpre (contraction over the rows)
                tn = torch.empty(lib.agcn_gemm_tn_scratch_bytes(M, Kd, N, 1), dtype=torch.uint8, device=dev)
                # d beta = <dpre, A W> = <A^T dpre, W> is a sum with heavy cancellation: when it is wanted, the
                # contraction runs in plain fp32 FMAs (tensor-core accumulation truncates) and the dot in double;
                # otherwise on the library's engine (-1), the one agcn_stack_loss_grad uses for BlockEnd
                want_dscale = has_scale and ctx.needs_input_grad[3]
                _lib.check(lib.agcn_gemm_tn(_ptr(A), None, _ptr(dpre), _ptr(dWu), M, Kd, N, 1, _ptr(tn),
                                            0 if want_dscale else -1, _stream_ptr(dev)))
                if want_dscale:
                    dscale = (dWu.double() * W.double()).sum().float().reshape(scale.shape)
                dW = dWu * scale if has_scale else dWu
        if has_bias and ctx.needs_input_grad[2]:
            dbias = dpre.sum(0)
        dadd = dpre if (has_add and ctx.needs_input_grad[4]) else None
        return dA, dW, dbias, dscale, dadd, None


def node_linear(A, W, bias=None, scale=None, add=None, activation="linear"):
    """[R, Fin] x [Fin, Fout] over all packed rows: act(scale * A W + bias + add).  activation in {linear, relu}."""
    return _NodeLinear.apply(A, W, bias, scale, add, activation)
