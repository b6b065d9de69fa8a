// A stack of SGC_LL layers + DenseMol + GraphGatherMol + logits + loss as ONE host call, its forward-only prediction
// call, and the Adam update.
//
// The reference runs a training step as one `sess.run([train_op, loss, ...])`
// (models/tf_modules/multitask_classifier.py:255-264): the TensorFlow runtime walks the whole graph of
// basic_AGCN.py:35-47 (4 x SGC_LL, DenseMol, GraphGatherMol, multitask logits, loss, AdamOptimizer) in C++ without
// returning to Python between layers.  agcn_stack_loss_grad is that call for this library: it chains
// agcn_sgcll_forward / agcn_head_loss_grad_ex / agcn_sgcll_backward -- the very entry points the layer classes
// use -- over one caller-provided arena, so a step costs one FFI crossing instead of ~10 autograd nodes with
// their allocations.  Nothing new is computed here; the kernels are the ones of the per-layer entry points.
#include <algorithm>
#include <cmath>
#include <vector>

#include "agcn_internal.cuh"

struct agcn_stack {
  std::vector<agcn_sgcll_desc> layers;
  int32_t Fm = 0, Nt = 0, loss_kind = 0;
  std::vector<int64_t> off;  // 5 per layer {weight, bias, M_L, alpha, beta | -1}, then dense_W, dense_b, head_W, head_b
};

namespace agcn {

// tf.train.AdamOptimizer (multitask_classifier.py:233-237):
//   lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t),  m = beta1 m + (1 - beta1) g,  v = beta2 v + (1 - beta2) g^2,
//   p -= lr_t m / (sqrt(v) + eps)
// t = *step + 1 is read from device memory, so a captured CUDA graph of the step replays with the right bias
// correction; adam_advance_kernel increments it afterwards.
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, const int32_t* __restrict__ step, long long n,
                                                   float lr, float beta1, float beta2, float eps) {
  __shared__ float s_lr_t;
  if (threadIdx.x == 0) {
    const double t = (double)(*step + 1);
    s_lr_t = (float)((double)lr * sqrt(1.0 - pow((double)beta2, t)) / (1.0 - pow((double)beta1, t)));
  }
  __syncthreads();
  const float lr_t = s_lr_t;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= lr_t * mi / (sqrtf(vi) + eps);
  }
}
__global__ void adam_advance_kernel(int32_t* step) { *step += 1; }

namespace {

inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

struct StackWork {
  std::vector<float*> H;      // activated output of layer l, [R, Fo_l]
  std::vector<void*> saved;   // forward -> backward area of layer l
  float* dA = nullptr;        // gradient ping-pong buffers [R, maxF]
  float* dB = nullptr;
  void* layer_work = nullptr;
  size_t layer_work_bytes = 0;
  void* head_work = nullptr;
  size_t head_work_bytes = 0;
  size_t bytes = 0;
};

int carve_stack(const agcn_stack* s, const agcn_plan* plan, void* base, StackWork* w) {
  char* b = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* r = b ? b + off : nullptr;
    off += al256(bytes);
    return r;
  };
  const size_t R = (size_t)plan->R;
  int maxF = 0;
  size_t work_max = 0;
  for (const agcn_sgcll_desc& d : s->layers) {
    size_t saved = 0, work = 0;
    int rc = agcn_sgcll_workspace_bytes(&d, plan, &saved, &work);
    if (rc) return rc;
    w->H.push_back(reinterpret_cast<float*>(take(R * d.Fo * sizeof(float))));
    w->saved.push_back(take(saved));
    work_max = std::max(work_max, work);
    maxF = std::max(maxF, std::max(d.F, d.Fo));
  }
  w->dA = reinterpret_cast<float*>(take(R * maxF * sizeof(float)));
  w->dB = reinterpret_cast<float*>(take(R * maxF * sizeof(float)));
  w->layer_work_bytes = work_max;
  w->layer_work = take(work_max);
  size_t hb = 0;
  int rc = agcn_head_workspace_bytes(plan, s->layers.back().Fo, s->Fm, s->Nt, &hb);
  if (rc) return rc;
  w->head_work_bytes = hb;
  w->head_work = take(hb);
  w->bytes = off;
  return AGCN_OK;
}

// Forward-only arena of agcn_stack_predict: nothing outlives a layer call, so two ping-pong activation buffers and one
// `saved` area (the layers run without AGCN_SAVE_FOR_BACKWARD; it is their forward scratch) serve every layer.
struct PredictWork {
  float* A = nullptr;  // activation ping-pong buffers [R, max Fo]
  float* B = nullptr;
  void* saved = nullptr;
  void* layer_work = nullptr;
  size_t layer_work_bytes = 0;
  void* head_work = nullptr;
  size_t head_work_bytes = 0;
  size_t bytes = 0;
};

agcn_sgcll_desc forward_only(const agcn_sgcll_desc& d) {
  agcn_sgcll_desc f = d;
  f.flags = 0;
  return f;
}

int carve_predict(const agcn_stack* s, const agcn_plan* plan, void* base, PredictWork* w) {
  char* b = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    void* r = b ? b + off : nullptr;
    off += al256(bytes);
    return r;
  };
  const size_t R = (size_t)plan->R;
  int maxFo = 0;
  size_t saved_max = 0, work_max = 0;
  for (const agcn_sgcll_desc& d : s->layers) {
    const agcn_sgcll_desc f = forward_only(d);
    size_t saved = 0, work = 0;
    int rc = agcn_sgcll_workspace_bytes(&f, plan, &saved, &work);
    if (rc) return rc;
    saved_max = std::max(saved_max, saved);
    work_max = std::max(work_max, work);
    maxFo = std::max(maxFo, d.Fo);
  }
  w->A = reinterpret_cast<float*>(take(R * maxFo * sizeof(float)));
  w->B = reinterpret_cast<float*>(take(R * maxFo * sizeof(float)));
  w->saved = take(saved_max);
  w->layer_work_bytes = work_max;
  w->layer_work = take(work_max);
  size_t hb = 0;
  int rc = agcn_head_predict_workspace_bytes(plan, s->layers.back().Fo, s->Fm, s->Nt, &hb);
  if (rc) return rc;
  w->head_work_bytes = hb;
  w->head_work = take(hb);
  w->bytes = off;
  return AGCN_OK;
}

}  // namespace
}  // namespace agcn

using namespace agcn;

extern "C" {

int agcn_stack_create(const agcn_sgcll_desc* layer_descs, int32_t n_layers, int32_t Fm, int32_t Nt, int32_t loss_kind,
                      const int64_t* param_offsets, agcn_stack** out) {
  AGCN_REQUIRE(layer_descs && n_layers >= 1 && param_offsets && out, "stack_create: bad arguments");
  AGCN_REQUIRE(Fm >= 1 && Nt >= 1, "stack_create: Fm and Nt must be positive");
  // the head calls take loss_kind as it is: agcn_stack_loss_grad / agcn_stack_predict need nothing per kind
  AGCN_REQUIRE(loss_kind == AGCN_LOSS_SIGMOID_CE || loss_kind == AGCN_LOSS_SOFTMAX_CE ||
                   loss_kind == AGCN_LOSS_WEIGHTED_L2,
               "stack_create: unknown loss_kind");
  for (int l = 0; l < n_layers; ++l) {
    AGCN_REQUIRE(layer_descs[l].variant == AGCN_VARIANT_SGC_LL, "stack_create: SGC_LL layers only (basic_AGCN.py:35-47)");
    AGCN_REQUIRE(l == 0 || layer_descs[l].F == layer_descs[l - 1].Fo, "stack_create: layer widths do not chain");
  }
  agcn_stack* s = new agcn_stack();
  s->layers.assign(layer_descs, layer_descs + n_layers);
  for (agcn_sgcll_desc& d : s->layers) d.flags = AGCN_SAVE_FOR_BACKWARD;
  s->Fm = Fm; s->Nt = Nt; s->loss_kind = loss_kind;
  s->off.assign(param_offsets, param_offsets + 5 * (size_t)n_layers + 4);
  *out = s;
  return AGCN_OK;
}

int agcn_stack_destroy(agcn_stack* s) {
  delete s;
  return AGCN_OK;
}

int agcn_stack_workspace_bytes(const agcn_stack* s, const agcn_plan* plan, size_t* bytes) {
  AGCN_REQUIRE(s && plan && bytes, "stack_workspace_bytes: null pointer");
  StackWork w;
  int rc = carve_stack(s, plan, nullptr, &w);
  if (rc) return rc;
  *bytes = w.bytes + 256;
  return AGCN_OK;
}

int agcn_stack_loss_grad(const agcn_stack* s, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                         const float* d_targets, const float* d_weights, float scale, const float* d_params,
                         float* d_grads, float* d_loss, void* d_work, size_t work_bytes, agcn_stack_notify_fn notify,
                         void* notify_user, void* stream) {
  AGCN_REQUIRE(s && plan && d_X && d_Lint && d_targets && d_weights && d_params && d_grads && d_loss && d_work,
               "stack_loss_grad: null pointer");
  StackWork w;
  int rc = carve_stack(s, plan, d_work, &w);
  if (rc) return rc;
  if (w.bytes > work_bytes) {
    set_error("stack_loss_grad: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  const int nl = (int)s->layers.size();
  auto P = [&](int l, int k) { return s->off[5 * (size_t)l + k] >= 0 ? d_params + s->off[5 * (size_t)l + k] : nullptr; };
  auto G = [&](int l, int k) { return s->off[5 * (size_t)l + k] >= 0 ? d_grads + s->off[5 * (size_t)l + k] : nullptr; };
  const int64_t* ho = &s->off[5 * (size_t)nl];
  // ---- forward (graphconv.py:85-125 per layer)
  const float* x = d_X;
  for (int l = 0; l < nl; ++l) {
    const agcn_sgcll_desc& d = s->layers[l];
    rc = agcn_sgcll_forward(&d, plan, x, d_Lint, nullptr, P(l, 2), P(l, 0), P(l, 1), P(l, 3), nullptr, w.H[l], nullptr,
                            nullptr, nullptr, w.saved[l], w.layer_work, w.layer_work_bytes, stream);
    if (rc) return rc;
    x = w.H[l];
  }
  // ---- DenseMol + GraphGatherMol + logits + loss, with every gradient of that part
  const agcn_sgcll_desc& last = s->layers[nl - 1];
  rc = agcn_head_loss_grad_ex(plan, w.H[nl - 1], d_params + ho[0], d_params + ho[1], d_params + ho[2], d_params + ho[3],
                              d_targets, d_weights, scale, s->loss_kind, last.Fo, s->Fm, s->Nt, d_loss, w.dA,
                              d_grads + ho[0], d_grads + ho[1], d_grads + ho[2], d_grads + ho[3], w.head_work,
                              w.head_work_bytes, stream);
  if (rc) return rc;
  if (notify) notify(notify_user, nl, stream);
  // ---- backward, last layer first; the first layer's input has no gradient unless the metric is differentiable
  float* dcur = w.dA;
  float* dnext = w.dB;
  for (int l = nl - 1; l >= 0; --l) {
    const agcn_sgcll_desc& d = s->layers[l];
    const bool full = d.laplacian_mode == AGCN_LAP_PAPER && d.metric_grad == AGCN_METRIC_GRAD_FULL;
    float* dX = (l > 0 || full) ? dnext : nullptr;
    rc = agcn_sgcll_backward(&d, plan, l == 0 ? d_X : w.H[l - 1], d_Lint, nullptr, P(l, 2), P(l, 0), P(l, 3), nullptr,
                             w.H[l], dcur, nullptr, w.saved[l], dX, G(l, 2), G(l, 0), G(l, 1), G(l, 3), nullptr, nullptr,
                             w.layer_work, w.layer_work_bytes, stream);
    if (rc) return rc;
    if (notify) notify(notify_user, l, stream);
    std::swap(dcur, dnext);
  }
  return AGCN_OK;
}

int agcn_stack_predict_workspace_bytes(const agcn_stack* s, const agcn_plan* plan, size_t* bytes) {
  AGCN_REQUIRE(s && plan && bytes, "stack_predict_workspace_bytes: null pointer");
  PredictWork w;
  int rc = carve_predict(s, plan, nullptr, &w);
  if (rc) return rc;
  *bytes = w.bytes + 256;
  return AGCN_OK;
}

int agcn_stack_predict(const agcn_stack* s, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                       const float* d_targets, const float* d_weights, float scale, const float* d_params,
                       float* d_probs, float* d_loss, void* d_work, size_t work_bytes, void* stream) {
  AGCN_REQUIRE(!d_targets == !d_weights && !d_targets == !d_loss,
               "stack_predict: d_targets, d_weights and d_loss must be all NULL or all set");
  AGCN_REQUIRE(s && plan && d_X && d_Lint && d_params && d_probs && d_work, "stack_predict: null pointer");
  PredictWork w;
  int rc = carve_predict(s, plan, d_work, &w);
  if (rc) return rc;
  if (w.bytes > work_bytes) {
    set_error("stack_predict: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  const int nl = (int)s->layers.size();
  auto P = [&](int l, int k) { return s->off[5 * (size_t)l + k] >= 0 ? d_params + s->off[5 * (size_t)l + k] : nullptr; };
  const int64_t* ho = &s->off[5 * (size_t)nl];
  const float* x = d_X;
  float* out = w.A;
  for (int l = 0; l < nl; ++l) {
    const agcn_sgcll_desc d = forward_only(s->layers[l]);
    rc = agcn_sgcll_forward(&d, plan, x, d_Lint, nullptr, P(l, 2), P(l, 0), P(l, 1), P(l, 3), nullptr, out, nullptr,
                            nullptr, nullptr, w.saved, w.layer_work, w.layer_work_bytes, stream);
    if (rc) return rc;
    x = out;
    out = out == w.A ? w.B : w.A;
  }
  return agcn_head_predict(plan, x, d_params + ho[0], d_params + ho[1], d_params + ho[2], d_params + ho[3], d_targets,
                           d_weights, scale, s->loss_kind, s->layers.back().Fo, s->Fm, s->Nt, d_probs, d_loss,
                           w.head_work, w.head_work_bytes, stream);
}

int agcn_adam_step(float* d_params, const float* d_grads, float* d_m, float* d_v, int32_t* d_step, int64_t n, float lr,
                   float beta1, float beta2, float eps, void* stream) {
  AGCN_REQUIRE(d_params && d_grads && d_m && d_v && d_step && n >= 1, "adam_step: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8);
  adam_kernel<<<blocks, 256, 0, st>>>(d_params, d_grads, d_m, d_v, d_step, (long long)n, lr, beta1, beta2, eps);
  AGCN_LAUNCH_CHECK();
  adam_advance_kernel<<<1, 1, 0, st>>>(d_step);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// ---- one graph launch per step (include/agcn_sgcll.h)
// A few executable graphs are kept, most recently used first: batches of a data set alternate between a handful of node
// topologies (which size buckets are populated, whether a graph above 144 nodes is present), and an in-place update only
// works against an executable graph of the same topology.
struct agcn_step_graph {
  static constexpr int KEEP = 4;
  cudaGraphExec_t exec[KEEP] = {nullptr, nullptr, nullptr, nullptr};
  // The captured graph whose parameters an executable graph was updated with stays alive until the launch that used them
  // has finished: objects a library attached to the capture (NCCL's plan of a captured collective) live as long as
  // that graph.  Ring of the last captures with an event behind their launch.
  static constexpr int RING = 3;
  cudaGraph_t src[RING] = {nullptr, nullptr, nullptr};
  cudaEvent_t done[RING] = {nullptr, nullptr, nullptr};
  int head = 0;
  long long instantiated = 0;
};

int agcn_capture_begin(void* stream) {
  AGCN_CUDA(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeThreadLocal));
  return AGCN_OK;
}

int agcn_capture_end_launch(void* stream, agcn_step_graph** graph, int32_t* how) {
  AGCN_REQUIRE(graph, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  cudaGraph_t g = nullptr;
  AGCN_CUDA(cudaStreamEndCapture(st, &g));
  if (!*graph) *graph = new agcn_step_graph();
  agcn_step_graph* sg = *graph;
  constexpr int KEEP = agcn_step_graph::KEEP;
  int hit = -1, why = 0;
  for (int i = 0; i < KEEP && hit < 0; ++i) {
    if (!sg->exec[i]) continue;
    cudaGraphExecUpdateResultInfo info;
    if (cudaGraphExecUpdate(sg->exec[i], g, &info) == cudaSuccess) {
      hit = i;
    } else {
      (void)cudaGetLastError();   // another node topology is not an error
      if (!why) why = (int)info.result;   // cudaGraphExecUpdateResult of the most recent executable graph
    }
  }
  cudaGraphExec_t use = nullptr;
  if (hit >= 0) {
    use = sg->exec[hit];
    for (int i = hit; i > 0; --i) sg->exec[i] = sg->exec[i - 1];
  } else {
    const cudaError_t e = cudaGraphInstantiate(&use, g, 0);
    if (e != cudaSuccess) {
      cudaGraphDestroy(g);
      AGCN_CUDA(e);
    }
    sg->instantiated++;
    if (sg->exec[KEEP - 1]) {   // evicted (rare): wait for its last launch before releasing it
      AGCN_CUDA(cudaStreamSynchronize(st));
      cudaGraphExecDestroy(sg->exec[KEEP - 1]);
    }
    for (int i = KEEP - 1; i > 0; --i) sg->exec[i] = sg->exec[i - 1];
  }
  sg->exec[0] = use;
  if (how) *how = hit >= 0 ? 1 : -why;
  AGCN_CUDA(cudaGraphLaunch(use, st));
  // retire the oldest capture of the ring (its launch was two steps ago), park this one behind its launch
  const int slot = sg->head;
  sg->head = (sg->head + 1) % agcn_step_graph::RING;
  if (sg->src[slot]) {
    AGCN_CUDA(cudaEventSynchronize(sg->done[slot]));
    cudaGraphDestroy(sg->src[slot]);
  }
  if (!sg->done[slot]) AGCN_CUDA(cudaEventCreateWithFlags(&sg->done[slot], cudaEventDisableTiming));
  sg->src[slot] = g;
  AGCN_CUDA(cudaEventRecord(sg->done[slot], st));
  return AGCN_OK;
}

int agcn_capture_abort(void* stream) {
  cudaGraph_t g = nullptr;
  (void)cudaStreamEndCapture((cudaStream_t)stream, &g);
  if (g) cudaGraphDestroy(g);
  (void)cudaGetLastError();
  return AGCN_OK;
}

int agcn_step_graph_destroy(agcn_step_graph* graph) {
  if (!graph) return AGCN_OK;
  (void)cudaDeviceSynchronize();   // a launch may still be in flight
  for (cudaGraphExec_t e : graph->exec)
    if (e) cudaGraphExecDestroy(e);
  for (int i = 0; i < agcn_step_graph::RING; ++i) {
    if (graph->src[i]) cudaGraphDestroy(graph->src[i]);
    if (graph->done[i]) cudaEventDestroy(graph->done[i]);
  }
  delete graph;
  return AGCN_OK;
}

}  // extern "C"
