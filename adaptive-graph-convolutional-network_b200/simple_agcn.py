"""SimpleAGCN-shaped training step used to MEASURE the SGC-LL hot path (bench.py) and to test it end to end.

The reference assembles the same stack in models/networks/basic_AGCN.py:35-47: four SGC_LL layers
(l_n_filters = [64, 128, 128, 64], utils/hyper_parameters.py:14), DenseMol, GraphGatherMol(tanh), then either
MultitaskGraphClassifier's per-task 2-class logits with weighted sigmoid cross-entropy divided by the batch size
(models/tf_modules/multitask_classifier.py:41-44,187-209) or SingletaskGraphClassifier's n_classes logits with
softmax cross-entropy (models/tf_modules/singletask_classifier.py:124-151) or MultitaskGraphRegressor's one output per
task with the weighted L2 divided by the batch size (models/tf_modules/multitask_regressor.py, DeepChem 1.x), and
tf.train.AdamOptimizer (multitask_classifier.py:233-237).  The reference executes one step as a single ``sess.run``; the counterpart
here is ONE library call, ``agcn_stack_loss_grad`` (engine="stack", the default and the path bench.py times),
which chains the same C entry points the layer classes use.  engine="autograd" runs the same step through the
layer classes and torch.autograd (the drop-in path of models/layers); tests pin both against the oracle and
against each other.

Data parallel: every rank holds a replica and its own shard of graphs; the flat gradient buffer is all-reduced
(SURVEY.md section 8e) -- in buckets issued while the earlier layers are still running backward when
``overlap_allreduce`` is set.  The loss is normalised by the GLOBAL batch size.
"""
import ctypes

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .batch import GraphBatch, PackedLaplacians, PackedNodes, _ptr, _stream_ptr
from .data_parallel import FlatGradBuffer, FlatParamBuffer
from .layers import SGC_LL
from .layers import graphconv as _gc


class SimpleAGCNStep(object):
    def __init__(self, n_feat=75, filters=(64, 128, 128, 64), final_feature_n=256, n_tasks=12, K=3, batch_size=256,
                 learning_rate=2e-3, device="cuda", world_size=1, laplacian="reference_literal",
                 metric_grad="reference", seed=123, loss="sigmoid_ce", engine="stack", overlap_allreduce=False,
                 beta1=0.9, beta2=0.999, epsilon=1e-8):
        """loss="sigmoid_ce": n_tasks two-class heads (Nt = 2 n_tasks logits);  loss="softmax_ce": one head with
        n_tasks classes (Nt = n_tasks logits);  loss="weighted_l2": n_tasks regression outputs (Nt = n_tasks),
        loss = sum (w (x - y))^2 / global batch."""
        if engine not in ("stack", "autograd"):
            raise ValueError("engine must be 'stack' or 'autograd'")
        if loss not in _lib.LOSS:
            raise ValueError("loss must be one of %s" % sorted(_lib.LOSS))
        self.device = torch.device(device)
        self.world_size = world_size
        self.global_batch = batch_size * world_size
        self.n_tasks = n_tasks
        self.loss_kind = loss
        self.engine = engine
        self.overlap_allreduce = overlap_allreduce and world_size > 1
        self.lr, self.beta1, self.beta2, self.epsilon = learning_rate, beta1, beta2, epsilon
        self.Nt = 2 * n_tasks if loss == "sigmoid_ce" else n_tasks
        self.Fm = final_feature_n
        if final_feature_n < 32 or final_feature_n % 4:
            raise ValueError("final_feature_n must be >= 32 and a multiple of 4 (agcn_head_loss_grad)")
        torch.manual_seed(seed)  # identical replicas on every rank
        _gc.DEFAULT_DEVICE[0] = str(self.device)
        self._build_layers(n_feat, filters, batch_size, K, laplacian, metric_grad)
        for l in self.layers:
            l.build()
        lim = float(np.sqrt(6.0 / (filters[-1] + final_feature_n)))
        self.dense_W = ((torch.rand(filters[-1], final_feature_n) * 2 - 1) * lim).to(self.device).requires_grad_(True)
        self.dense_b = torch.zeros(final_feature_n, device=self.device, requires_grad=True)
        # n_tasks independent [n_feature, 2] logits heads == one [n_feature, 2 * n_tasks] matrix
        self.head_W = torch.nn.init.trunc_normal_(torch.empty(final_feature_n, self.Nt), std=0.01, a=-0.02,
                                                  b=0.02).to(self.device).requires_grad_(True)
        self.head_b = torch.zeros(self.Nt, device=self.device, requires_grad=True)
        self.params = [v for l in self.layers for v in l.vars.values()] + [self.dense_W, self.dense_b, self.head_W,
                                                                           self.head_b]
        # one flat gradient buffer and one flat parameter buffer; every parameter / .grad is a view into them, and every
        # producer (SGC-LL backward, head) OVERWRITES its gradients in place: nothing to zero, nothing to accumulate
        self.grads = FlatGradBuffer(self.params, direct=self.params)
        self.flat_grad = self.grads.flat
        self.flat_params = FlatParamBuffer(self.params, self.grads)
        self.adam_m = torch.zeros_like(self.flat_grad)
        self.adam_v = torch.zeros_like(self.flat_grad)
        self.adam_step = torch.zeros(1, dtype=torch.int32, device=self.device)
        # offsets of every tensor in the flat buffers (the layout agcn_stack_create takes)
        offs, off = [], 0
        self._stage_slices = []
        for l in self.layers:
            start = off
            per = {}
            for name, v in l.vars.items():
                per[name] = off
                off += v.numel()
            offs += [per.get(k, -1) for k in ("weight", "bias", "M_L", "alpha", "beta")]
            self._stage_slices.append((start, off))
        start = off
        for t in (self.dense_W, self.dense_b, self.head_W, self.head_b):
            offs.append(off)
            off += t.numel()
        self._stage_slices.append((start, off))      # stage n_layers = dense + head
        assert off == self.flat_grad.numel()
        self._stack = ctypes.c_void_p()
        self._create_stack((ctypes.c_int64 * len(offs))(*offs))
        self._arena = None
        self._pred_arena = None
        self._step_graph = ctypes.c_void_p()
        self._graph_stream = None
        # opt-in: capture the NCCL all-reduce of the multi-GPU step too (launched by torch.distributed on its own stream,
        # which the events of ProcessGroupNCCL fork from and join back into the capturing stream)
        self.graph_collectives = False
        self._graph_miss_streak = 0
        self._graph_disabled = False
        self.step_graph_refusals = []   # cudaGraphExecUpdateResult codes of the steps that had to instantiate
        self.step_graph_updates = 0     # steps whose executable graph was updated in place (not instantiated anew)
        self._loss = torch.zeros(1, device=self.device, dtype=torch.float32)
        self._pending = []
        self._notify = _lib.NOTIFY_FN(self._on_stage)     # keep the ctypes thunk alive

    # ---- the body of the network (ResAGCNStep overrides these three) ---------------------------------------------
    def _build_layers(self, n_feat, filters, batch_size, K, laplacian, metric_grad):
        """self.layers, in the order of the flat buffers (basic_AGCN.py:35-45: SGC_LL layers with relu)."""
        dims = [n_feat] + list(filters)
        self.layers = [SGC_LL(dims[i + 1], dims[i], batch_size, K=K, activation='relu', laplacian=laplacian,
                              metric_grad=metric_grad) for i in range(len(filters))]

    def _create_stack(self, offs):
        """self._stack from the layers and the flat-buffer offsets (5 per layer, then the 4 head tensors)."""
        descs = (_lib.Desc * len(self.layers))()
        for i, l in enumerate(self.layers):
            descs[i] = _layer_desc(l)
        _lib.check(_lib.lib().agcn_stack_create(descs, len(self.layers), self.Fm, self.Nt, _lib.LOSS[self.loss_kind],
                                                offs, ctypes.byref(self._stack)))

    def _body(self, x):
        """The layer classes on the input dict of the drop-in path -> PackedNodes output of the last layer."""
        for layer in self.layers:
            out, _, _ = layer(x)
            x = dict(x, node_features=out)
        return out

    def __del__(self):
        try:
            if self._step_graph:
                _lib.lib().agcn_step_graph_destroy(self._step_graph)
                self._step_graph = ctypes.c_void_p()
            if self._stack:
                _lib.lib().agcn_stack_destroy(self._stack)
                self._stack = ctypes.c_void_p()
        except Exception:
            pass

    def n_parameters(self):
        return int(self.flat_grad.numel())

    # ---- gradient exchange ----------------------------------------------------------------------------------
    def _on_stage(self, _user, stage, _stream):
        """agcn_stack_notify_fn: the gradients of `stage` are enqueued -> start the all-reduce of that bucket on
        NCCL's stream while the earlier layers run backward."""
        a, b = self._stage_slices[stage]
        self._pending.append(dist.all_reduce(self.flat_grad[a:b], async_op=True))

    def _all_reduce(self):
        if self.world_size <= 1:
            return
        if self.overlap_allreduce and self.engine == "stack":
            for w in self._pending:
                w.wait()                        # stream-level wait: Adam is ordered after every bucket
            self._pending = []
        else:
            self.grads.all_reduce()

    # ---- engines --------------------------------------------------------------------------------------------
    def _ensure_arena(self, batch, predict=False):
        """The device arena of agcn_stack_loss_grad (self._arena) or, predict=True, of agcn_stack_predict
        (self._pred_arena) for this batch: grown with 25 % headroom when it is too small, reused otherwise."""
        lib = _lib.lib()
        size_fn, attr = ((lib.agcn_stack_predict_workspace_bytes, "_pred_arena") if predict else
                         (lib.agcn_stack_workspace_bytes, "_arena"))
        nbytes = ctypes.c_size_t()
        _lib.check(size_fn(self._stack, batch.handle, ctypes.byref(nbytes)))
        arena = getattr(self, attr)
        if arena is None or arena.numel() < nbytes.value:
            arena = torch.empty(int(nbytes.value * 1.25) + 4096, dtype=torch.uint8, device=self.device)
            setattr(self, attr, arena)
        return arena

    def _loss_grad_stack(self, X, Lint, batch, targets, weights):
        lib = _lib.lib()
        arena = self._ensure_arena(batch)
        notify = ctypes.cast(self._notify, ctypes.c_void_p) if self.overlap_allreduce else None
        with torch.cuda.device(self.device):
            _lib.check(lib.agcn_stack_loss_grad(
                self._stack, batch.handle, _ptr(X), _ptr(Lint), _ptr(targets), _ptr(weights),
                1.0 / self.global_batch, _ptr(self.flat_params.flat), _ptr(self.flat_grad), _ptr(self._loss),
                _ptr(arena), arena.numel(), notify, None, _stream_ptr(self.device)))
        return self._loss

    def forward_loss(self, X, Lint, batch, targets, weights):
        """The drop-in path: layer classes + torch.autograd.  X [R, F] packed, Lint packed, targets [B, Nt] float,
        weights [B, Nt] (sigmoid_ce, weighted_l2) or [B] (softmax_ce) -> scalar loss."""
        from .functional import head_loss
        x = {'node_features': PackedNodes(X, batch), 'original_laplacian': PackedLaplacians(Lint, batch),
             'data_slice': None, 'lap_slice': None, '_batch': batch}
        out = self._body(x)
        return head_loss(out.data, self.dense_W, self.dense_b, self.head_W, self.head_b, targets, weights, batch,
                         1.0 / self.global_batch, unit_grad=True, loss_kind=self.loss_kind)

    def loss_and_grads(self, X, Lint, batch, targets, weights):
        """Loss (1-element tensor) with every gradient written into the flat gradient buffer (not yet reduced)."""
        X, Lint = X.contiguous(), Lint.contiguous()
        targets, weights = targets.contiguous(), weights.contiguous()
        assert X.shape[0] == batch.total_nodes and Lint.numel() == batch.total_lap
        assert targets.shape == (batch.batch_size, self.Nt)
        if self.engine == "stack":
            return self._loss_grad_stack(X, Lint, batch, targets, weights)
        loss = self.forward_loss(X, Lint, batch, targets, weights)
        loss.backward()
        return loss.detach().reshape(1)

    # ---- prediction (predict_proba / predict / evaluate of the reference's classifiers and regressor) ------------
    def _predict_stack(self, X, Lint, batch, targets, weights, scale):
        lib = _lib.lib()
        arena = self._ensure_arena(batch, predict=True)
        probs = torch.empty(batch.batch_size, self.Nt, device=self.device, dtype=torch.float32)
        loss = torch.empty(1, device=self.device, dtype=torch.float32) if targets is not None else None
        with torch.cuda.device(self.device):
            _lib.check(lib.agcn_stack_predict(
                self._stack, batch.handle, _ptr(X), _ptr(Lint), _ptr(targets), _ptr(weights),
                float(scale if scale is not None else 0.0), _ptr(self.flat_params.flat), _ptr(probs), _ptr(loss),
                _ptr(arena), arena.numel(), _stream_ptr(self.device)))
        return probs, (loss.reshape(()) if loss is not None else None)

    def _predict(self, X, Lint, batch, targets=None, weights=None, scale=None):
        """(probs [B, Nt] -- the values for weighted_l2 --, loss or None) of the current parameters; no gradient, no
        parameter or optimizer state touched."""
        X, Lint = X.contiguous(), Lint.contiguous()
        assert X.shape[0] == batch.total_nodes and Lint.numel() == batch.total_lap
        if targets is not None:
            targets, weights = targets.contiguous(), weights.contiguous()
            assert targets.shape == (batch.batch_size, self.Nt)
            scale = 1.0 / batch.batch_size if scale is None else scale
        if self.engine == "stack":
            return self._predict_stack(X, Lint, batch, targets, weights, scale)
        from .functional import head_predict
        x = {'node_features': PackedNodes(X, batch), 'original_laplacian': PackedLaplacians(Lint, batch),
             'data_slice': None, 'lap_slice': None, '_batch': batch}
        with torch.no_grad():
            out = self._body(x)
            return head_predict(out.data, self.dense_W, self.dense_b, self.head_W, self.head_b, batch, self.loss_kind,
                                targets, weights, scale)

    def _shape_probs(self, probs):
        return probs.reshape(probs.shape[0], -1, 2) if self.loss_kind == "sigmoid_ce" else probs

    def predict_proba(self, X, Lint, batch):
        """Class probabilities: [B, n_tasks, 2] for sigmoid_ce (softmax over each task's two logits), [B, n_classes]
        for softmax_ce.  X [R, F] packed, Lint packed.  A weighted_l2 regressor has none: ValueError (use predict)."""
        if self.loss_kind == "weighted_l2":
            raise ValueError("predict_proba: a regressor (loss='weighted_l2') has no class probabilities; use predict")
        return self._shape_probs(self._predict(X, Lint, batch)[0])

    def predict(self, X, Lint, batch):
        """Class labels (int64): [B, n_tasks] for sigmoid_ce, [B] for softmax_ce.  weighted_l2: the regression values
        (float32) [B, n_tasks]."""
        if self.loss_kind == "weighted_l2":
            return self._predict(X, Lint, batch)[0]
        return self.predict_proba(X, Lint, batch).argmax(-1)

    def evaluate(self, X, Lint, batch, targets, weights, scale=None):
        """(probabilities as predict_proba -- the values as predict for weighted_l2 --, loss): the loss is the training
        loss of this batch without its gradients, bit for bit what loss_and_grads returns with the same scale (default
        1 / batch size)."""
        if targets is None or weights is None:
            raise ValueError("evaluate needs targets and weights")
        probs, loss = self._predict(X, Lint, batch, targets, weights, scale)
        return self._shape_probs(probs), loss

    def apply_adam(self):
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().agcn_adam_step(
                _ptr(self.flat_params.flat), _ptr(self.flat_grad), _ptr(self.adam_m), _ptr(self.adam_v),
                _ptr(self.adam_step), self.flat_grad.numel(), self.lr, self.beta1, self.beta2, self.epsilon,
                _stream_ptr(self.device)))

    def step(self, X, Lint, batch, targets, weights):
        """One training step: forward, backward, gradient all-reduce, Adam.  Returns the loss (1-element tensor,
        valid until the next step)."""
        loss = self.loss_and_grads(X, Lint, batch, targets, weights)
        self._all_reduce()
        self.apply_adam()
        return loss


    def step_graphed(self, X, Lint, batch, targets, weights):
        """step() as ONE graph launch: the library calls of the step are captured (nothing runs, the host pays what the
        launches cost), the executable graph of the previous step is updated in place with the new batch's kernel
        parameters and launched (agcn_capture_begin / agcn_capture_end_launch).  For batches arriving over PCIe beside the
        step: eager launch commands are fetched from host memory one by one and bulk transfers delay every fetch.
        With more than one process the step stays eager unless graph_collectives is set (the NCCL all-reduce is launched
        by torch.distributed; captured with it: tools/e2e_multi.py)."""
        if self.engine != "stack" or self._graph_disabled or (self.world_size > 1 and not self.graph_collectives):
            return self.step(X, Lint, batch, targets, weights)
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream == 0 and self.world_size > 1:
            # (capturing the all-reduce on a borrowed stream hung under mp.spawn in the 2-rank test: unexplained, refused)
            raise RuntimeError("step_graphed with graph_collectives must be called on a non-default CUDA stream")
        if cur.cuda_stream == 0:            # the legacy default stream cannot be captured: borrow a stream of our own
            if self._graph_stream is None:
                self._graph_stream = torch.cuda.Stream(device=self.device)
            gs = self._graph_stream
            gs.wait_stream(cur)
            with torch.cuda.stream(gs):
                loss = self.step_graphed(X, Lint, batch, targets, weights)
            cur.wait_stream(gs)
            return loss
        lib = _lib.lib()
        self._ensure_arena(batch)           # no allocation inside the capture
        st = _stream_ptr(self.device)
        keep, self.overlap_allreduce = self.overlap_allreduce, False      # no host callbacks inside the capture
        try:
            with torch.cuda.device(self.device):
                _lib.check(lib.agcn_capture_begin(st))
                try:
                    loss = self.loss_and_grads(X, Lint, batch, targets, weights)
                    self._all_reduce()          # (graph_collectives: torch's NCCL all-reduce joins the capture)
                    self.apply_adam()
                except BaseException:
                    lib.agcn_capture_abort(st)
                    raise
                how = ctypes.c_int32(0)
                _lib.check(lib.agcn_capture_end_launch(st, ctypes.byref(self._step_graph), ctypes.byref(how)))
        finally:
            self.overlap_allreduce = keep
        if how.value == 1:
            self.step_graph_updates += 1
            self._graph_miss_streak = 0
        else:
            self.step_graph_refusals.append(int(-how.value))
            self._graph_miss_streak += 1
            if self._graph_miss_streak >= 4:
                # instantiating a graph costs several eager steps: a stream of batches that never matches a kept
                # executable graph goes back to eager launches for good
                self._graph_disabled = True
        return loss


def _layer_desc(layer):
    """agcn_sgcll_desc of an SGC_LL / SGC_LL_Reslap layer with a fused relu (the stack sets the flags)."""
    lap, mg = layer._semantics()
    return _lib.Desc(layer.n_atom_feature, layer.nb_filter, layer.K, _lib.VARIANT[layer.variant], _lib.LAPLACIAN[lap],
                     _lib.METRIC_GRAD[mg], _lib.ACT["relu"], _lib.SAVE_FOR_BACKWARD)


def expand_labels(y, w, targets, weights, stream=None):
    """Labels as the reference feeds them (multitask_classifier.py:147-152,171-185) -> the one-hot targets / per-logit
    weights of the sigmoid heads (tf.one_hot(label, 2), :196-199), on the device in one kernel.
    y: uint8 / bool [B, T], w: float32 [B, T]; CUDA tensors or PINNED host tensors (read in place over PCIe).
    targets, weights: float32 CUDA [B, 2T], overwritten.  The caller keeps y / w unchanged until the stream gets there."""
    B, T = y.shape
    for t in (y, w):
        if not t.is_cuda and not t.is_pinned():
            raise ValueError("host label tensors must be pinned (tensor.pin_memory()) to be read by the device")
    if y.dtype == torch.bool:
        y = y.view(torch.uint8)
    if y.dtype != torch.uint8 or w.dtype != torch.float32 or not y.is_contiguous() or not w.is_contiguous():
        raise ValueError("expand_labels: y must be contiguous uint8 / bool, w contiguous float32")
    if targets.shape != (B, 2 * T) or weights.shape != (B, 2 * T) or not targets.is_cuda or not weights.is_cuda:
        raise ValueError("expand_labels: targets / weights must be CUDA [B, 2T]")
    dev = targets.device
    with torch.cuda.device(dev):
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        _lib.check(_lib.lib().agcn_expand_labels(ctypes.c_void_p(y.data_ptr()), ctypes.c_void_p(w.data_ptr()), B, T,
                                                 _ptr(targets), _ptr(weights), ctypes.c_void_p(st.cuda_stream)))
    return targets, weights


def synthetic_labels(B, n_tasks, seed, device, loss="sigmoid_ce"):
    """sigmoid_ce: Bernoulli(0.1) labels as one-hot float targets [B, 2T], weights [B, 2T] = 1 (SURVEY.md 8d).
    softmax_ce: uniform class labels as one-hot [B, T], per-sample weights [B] = 1.
    weighted_l2: N(0, 1) targets [B, T], 0/1 weights [B, T] with about 10 % zeros (missing labels)."""
    rng = np.random.default_rng(seed)
    if loss == "weighted_l2":
        y = rng.standard_normal((B, n_tasks)).astype(np.float32)
        w = (rng.random((B, n_tasks)) >= 0.1).astype(np.float32)
        return torch.from_numpy(y).to(device), torch.from_numpy(w).to(device)
    if loss == "softmax_ce":
        y = rng.integers(0, n_tasks, B)
        onehot = np.zeros((B, n_tasks), np.float32)
        onehot[np.arange(B), y] = 1.0
        return torch.from_numpy(onehot).to(device), torch.ones(B, dtype=torch.float32).to(device)
    y = (rng.random((B, n_tasks)) < 0.1)
    onehot = np.zeros((B, n_tasks, 2), np.float32)
    onehot[..., 0] = ~y
    onehot[..., 1] = y
    w = np.ones((B, 2 * n_tasks), np.float32)
    return torch.from_numpy(onehot.reshape(B, 2 * n_tasks)).to(device), torch.from_numpy(w).to(device)
