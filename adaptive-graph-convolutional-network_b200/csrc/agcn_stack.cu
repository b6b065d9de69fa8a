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
//
// A stack is a list of nodes (agcn_stack_create_nodes): SGC_LL layers, SGC_LL_Reslap layers whose L_prev is an earlier
// Reslap layer's L_all (ResidualGraphMolResLap, tf_graphs.py:159-223), and BlockEnd nodes that close a residual block
// (blockend.py:67-86, through agcn_node_gemm / agcn_gemm_tn as functional._NodeLinear calls them).
// agcn_stack_create is the list of SGC_LL layers.
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "agcn_internal.cuh"

struct agcn_stack {
  std::vector<agcn_stack_node> nodes;  // desc.flags as the layer classes set them
  int32_t Fm = 0, Nt = 0, loss_kind = 0;
  std::vector<int64_t> off;  // 5 per node {weight, bias, M_L, alpha, beta | -1}, then dense_W, dense_b (-1, -1 for the
                             // per-node head), head_W, head_b
  // topology, derived once by agcn_stack_create_nodes
  std::vector<int32_t> lall_user;   // Reslap node i: the Reslap node whose L_prev is L_all[i], or -1
  std::vector<int32_t> res_user;    // node i: the BlockEnd whose x_res is H[i], or -1
  // agcn_stack_predict: slot of the activation buffer each node writes, slot of the L_all each Reslap node writes
  std::vector<int32_t> pred_h, pred_l;
  int32_t n_pred_h = 0, n_pred_l = 0;
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

// BlockEnd backward: dpre = dY * act'(Y), written as functional._NodeLinear writes it (dC * (C > 0) for relu, a copy of
// dC for linear), so that the stack and the layer classes feed bit-identical operands to the products that follow.
__global__ void __launch_bounds__(256) act_grad_kernel(const float* __restrict__ dY, const float* __restrict__ Y,
                                                       float* __restrict__ dpre, long long n, int relu) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dpre[i] = relu ? dY[i] * (Y[i] > 0.f ? 1.f : 0.f) : dY[i];
}

namespace {

bool is_reslap(const agcn_stack_node& n) {
  return n.kind == AGCN_NODE_SGCLL && n.desc.variant == AGCN_VARIANT_SGC_LL_RESLAP;
}

// flags of a layer in agcn_stack_predict: no SAVE_FOR_BACKWARD (the `saved` area is forward scratch), the rest as in
// training, so that every layer takes the same kernels in both calls
agcn_sgcll_desc forward_only(const agcn_sgcll_desc& d) {
  agcn_sgcll_desc f = d;
  f.flags &= ~AGCN_SAVE_FOR_BACKWARD;
  return f;
}

// `saved` and scratch bytes of node i's forward (train) or forward-only call; a BlockEnd saves nothing, its scratch
// serves agcn_node_gemm forward / dX (sized as functional._NodeLinear sizes it) and the TN dW
int node_bytes(const agcn_stack_node& nd, const agcn_plan* plan, bool train, size_t* saved, size_t* work) {
  const agcn_sgcll_desc& d = nd.desc;
  *saved = 0;
  if (nd.kind == AGCN_NODE_SGCLL) {
    const agcn_sgcll_desc f = train ? d : forward_only(d);
    return agcn_sgcll_workspace_bytes(&f, plan, saved, work);
  }
  const int m = std::max(d.F, d.Fo);
  *work = std::max(agcn_node_gemm_scratch_bytes(m, m), agcn_gemm_tn_scratch_bytes((int32_t)plan->R, d.F, d.Fo, 1));
  return AGCN_OK;
}

bool node_head(const agcn_stack* s) { return s->loss_kind == AGCN_PER_NODE_SOFTMAX_CE; }

// work area of the head call of agcn_stack_loss_grad (train) or agcn_stack_predict
int head_bytes(const agcn_stack* s, const agcn_plan* plan, bool train, size_t* bytes) {
  const int32_t Fh = s->nodes.back().desc.Fo;
  if (node_head(s))
    return train ? agcn_node_head_workspace_bytes(plan, Fh, s->Nt, bytes)
                 : agcn_node_head_predict_workspace_bytes(plan, Fh, s->Nt, bytes);
  return train ? agcn_head_workspace_bytes(plan, Fh, s->Fm, s->Nt, bytes)
               : agcn_head_predict_workspace_bytes(plan, Fh, s->Fm, s->Nt, bytes);
}

// Where the forward walk finds node i's output, L_all and `saved` area, and the scratch of the layer and head calls.
// Training gives every node areas of its own; prediction points the nodes at reused slots and one shared `saved` area.
struct StackWork {
  std::vector<float*> H;      // activated output of node i, [R, Fo_i]
  std::vector<float*> Lall;   // Reslap node i: its L_all [sum n^2]
  std::vector<void*> saved;   // SGC-LL node i: its forward -> backward area (prediction: forward scratch)
  void* layer_work = nullptr;
  size_t layer_work_bytes = 0;
  void* head_work = nullptr;
  size_t head_work_bytes = 0;
  // training only
  float* dA = nullptr;        // gradient ping-pong buffers [R, maxF]
  float* dB = nullptr;
  std::vector<float*> dLall;  // Reslap node i with a consumer: gradient into L_all[i] [sum n^2]
  std::vector<float*> dpre;   // BlockEnd node i: dY * act'(Y) [R, Fo_i], alive until its dX product has run
  size_t bytes = 0;
};

// A plain SGC_LL stack (agcn_stack_create) carves exactly the areas it always had, in the same order; the Reslap and
// BlockEnd areas come after them.
int carve_stack(const agcn_stack* s, const agcn_plan* plan, void* base, StackWork* w) {
  Arena c(base);
  const size_t R = (size_t)plan->R, LL = (size_t)plan->LL;
  const int n = (int)s->nodes.size();
  int maxF = 0;
  size_t work_max = 0;
  for (const agcn_stack_node& nd : s->nodes) {
    size_t saved = 0, work = 0;
    int rc = node_bytes(nd, plan, true, &saved, &work);
    if (rc) return rc;
    w->H.push_back(c.take(R * nd.desc.Fo));
    w->saved.push_back(nd.kind == AGCN_NODE_SGCLL ? c.area(saved) : nullptr);
    work_max = std::max(work_max, work);
    maxF = std::max(maxF, std::max(nd.desc.F, nd.desc.Fo));
  }
  w->dA = c.take(R * maxF);
  w->dB = c.take(R * maxF);
  w->layer_work_bytes = work_max;
  w->layer_work = c.area(work_max);
  int rc = head_bytes(s, plan, true, &w->head_work_bytes);
  if (rc) return rc;
  w->head_work = c.area(w->head_work_bytes);
  w->Lall.assign(n, nullptr);
  w->dLall.assign(n, nullptr);
  w->dpre.assign(n, nullptr);
  for (int i = 0; i < n; ++i) {
    const agcn_stack_node& nd = s->nodes[i];
    if (is_reslap(nd)) {
      w->Lall[i] = c.take(LL);
      if (s->lall_user[i] >= 0) w->dLall[i] = c.take(LL);
    } else if (nd.kind == AGCN_NODE_BLOCK_END) {
      w->dpre[i] = c.take(R * nd.desc.Fo);
    }
  }
  w->bytes = c.bytes;
  return AGCN_OK;
}

// Forward-only arena of agcn_stack_predict: one `saved` area serves every layer (the layers run without
// AGCN_SAVE_FOR_BACKWARD; it is their forward scratch), and the activations and L_all matrices live in slots that are
// reused as soon as their last reader has run (agcn_stack_create_nodes assigns them).  A plain SGC_LL stack gets two
// activation slots, used alternately, and no L_all slot.
int carve_predict(const agcn_stack* s, const agcn_plan* plan, void* base, StackWork* w) {
  Arena c(base);
  const size_t R = (size_t)plan->R;
  const int n = (int)s->nodes.size();
  int maxFo = 0;
  size_t saved_max = 0, work_max = 0;
  for (const agcn_stack_node& nd : s->nodes) {
    size_t saved = 0, work = 0;
    int rc = node_bytes(nd, plan, false, &saved, &work);
    if (rc) return rc;
    saved_max = std::max(saved_max, saved);
    work_max = std::max(work_max, work);
    maxFo = std::max(maxFo, nd.desc.Fo);
  }
  std::vector<float*> h_slot, l_slot;
  for (int k = 0; k < s->n_pred_h; ++k) h_slot.push_back(c.take(R * maxFo));
  void* saved = c.area(saved_max);
  w->layer_work_bytes = work_max;
  w->layer_work = c.area(work_max);
  int rc = head_bytes(s, plan, false, &w->head_work_bytes);
  if (rc) return rc;
  w->head_work = c.area(w->head_work_bytes);
  for (int k = 0; k < s->n_pred_l; ++k) l_slot.push_back(c.take((size_t)plan->LL));
  for (int i = 0; i < n; ++i) {
    const bool sgcll = s->nodes[i].kind == AGCN_NODE_SGCLL;
    w->H.push_back(h_slot[s->pred_h[i]]);
    w->Lall.push_back(s->pred_l[i] >= 0 ? l_slot[s->pred_l[i]] : nullptr);
    w->saved.push_back(sgcll ? saved : nullptr);
  }
  w->bytes = c.bytes;
  return AGCN_OK;
}

// Greedy slot assignment over the node order: value i is written by node i and read for the last time by node
// last[i]; it takes the lowest slot whose value has had its last read before node i (a node's inputs stay untouched
// while it writes its output).  want[i] = false: node i writes no value.
int assign_slots(const std::vector<int32_t>& last, const std::vector<bool>& want, std::vector<int32_t>* slot) {
  std::vector<int32_t> busy_until;   // per slot: last reader of the value it holds
  slot->assign(last.size(), -1);
  for (size_t i = 0; i < last.size(); ++i) {
    if (!want[i]) continue;
    int k = 0;
    while (k < (int)busy_until.size() && busy_until[k] >= (int32_t)i) ++k;
    if (k == (int)busy_until.size()) busy_until.push_back(0);
    busy_until[k] = last[i];
    (*slot)[i] = k;
  }
  return (int)busy_until.size();
}

// forward of BlockEnd node i (blockend.py:67-86) as functional._NodeLinear runs it: C = H[i-1], then
// C += H[src] W with the activation in the product's epilogue
int block_end_forward(const agcn_sgcll_desc& d, const agcn_plan* plan, const float* x, const float* x_res,
                      const float* W, float* out, void* work, cudaStream_t st) {
  const int32_t R = (int32_t)plan->R;
  AGCN_CUDA(cudaMemcpyAsync(out, x, (size_t)R * d.Fo * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return agcn_node_gemm(x_res, d.F, W, d.Fo, 0, out, d.Fo, R, d.Fo, d.F, nullptr, nullptr, 1, d.activation, work, st);
}

// tensor k of node l's parameters (k: weight, bias, M_L, alpha, beta) in a flat buffer, NULL when the node has none
template <typename T>
T* node_param(const agcn_stack* s, T* flat, int l, int k) {
  const int64_t o = s->off[5 * (size_t)l + k];
  return o >= 0 ? flat + o : nullptr;
}

// The forward of every node (graphconv.py:85-125 / graphconv_reslap.py:45-89 per layer, blockend.py:67-86 per
// BlockEnd) into the areas `w` names for it; train: the layers save what their backward needs.
int forward_nodes(const agcn_stack* s, const agcn_plan* plan, const StackWork& w, const float* d_X, const float* d_Lint,
                  const float* d_params, bool train, void* stream) {
  const float* x = d_X;
  for (int l = 0; l < (int)s->nodes.size(); ++l) {
    const agcn_stack_node& nd = s->nodes[l];
    const agcn_sgcll_desc d = train ? nd.desc : forward_only(nd.desc);
    auto P = [&](int k) { return node_param(s, d_params, l, k); };
    int rc;
    if (nd.kind == AGCN_NODE_BLOCK_END) {
      rc = block_end_forward(d, plan, x, w.H[nd.src], P(0), w.H[l], w.layer_work, (cudaStream_t)stream);
    } else {
      const float* Lprev = (is_reslap(nd) && nd.src >= 0) ? w.Lall[nd.src] : nullptr;
      rc = agcn_sgcll_forward(&d, plan, x, d_Lint, Lprev, P(2), P(0), P(1), P(3), P(4), w.H[l], nullptr, nullptr,
                              w.Lall[l], w.saved[l], w.layer_work, w.layer_work_bytes, stream);
    }
    if (rc) return rc;
    x = w.H[l];
  }
  return AGCN_OK;
}

}  // namespace
}  // namespace agcn

using namespace agcn;

extern "C" {

int agcn_stack_create_nodes(const agcn_stack_node* nodes, int32_t n_nodes, int32_t Fm, int32_t Nt, int32_t loss_kind,
                            const int64_t* param_offsets, agcn_stack** out) {
  AGCN_REQUIRE(nodes && n_nodes >= 1 && param_offsets && out, "stack_create: bad arguments");
  *out = nullptr;
  const bool per_node = loss_kind == AGCN_PER_NODE_SOFTMAX_CE;
  AGCN_REQUIRE(per_node || (Fm >= 1 && Nt >= 1), "stack_create: Fm and Nt must be positive");
  // the graph-head calls take loss_kind as it is: agcn_stack_loss_grad / agcn_stack_predict need nothing per kind
  // beyond choosing between them and the per-node head
  AGCN_REQUIRE(loss_kind == AGCN_LOSS_SIGMOID_CE || loss_kind == AGCN_LOSS_SOFTMAX_CE ||
                   loss_kind == AGCN_LOSS_WEIGHTED_L2 || per_node,
               "stack_create: unknown loss_kind");
  if (per_node) {
    AGCN_REQUIRE(Fm == 0 && Nt >= 1, "stack_create: the per-node head has no DenseMol (Fm must be 0) and Nt >= 1 classes");
    AGCN_REQUIRE(param_offsets[5 * (size_t)n_nodes] == -1 && param_offsets[5 * (size_t)n_nodes + 1] == -1,
                 "stack_create: the per-node head has no dense_W / dense_b (their offsets must be -1)");
  }
  std::vector<int32_t> lall_user(n_nodes, -1), res_user(n_nodes, -1);
  for (int i = 0; i < n_nodes; ++i) {
    const agcn_stack_node& nd = nodes[i];
    const agcn_sgcll_desc& d = nd.desc;
    const std::string at = "stack_create_nodes: node " + std::to_string(i) + ": ";
    AGCN_REQUIRE(nd.kind == AGCN_NODE_SGCLL || nd.kind == AGCN_NODE_BLOCK_END, at + "unknown kind");
    if (nd.kind == AGCN_NODE_BLOCK_END) {
      AGCN_REQUIRE(i > 0, at + "a BlockEnd cannot be the first node (it adds to the previous node's output)");
      AGCN_REQUIRE(nd.src >= 0 && nd.src < i, at + "src must be an earlier node");
      AGCN_REQUIRE(res_user[nd.src] < 0, at + "two BlockEnds name the same src");
      AGCN_REQUIRE(d.F == nodes[nd.src].desc.Fo && d.Fo == nodes[i - 1].desc.Fo,
                   at + "widths do not chain (F must be the width of H[src], Fo the width of H[i-1])");
      res_user[nd.src] = i;
      continue;
    }
    AGCN_REQUIRE(d.variant == AGCN_VARIANT_SGC_LL || d.variant == AGCN_VARIANT_SGC_LL_RESLAP, at + "unknown variant");
    AGCN_REQUIRE(i == 0 || d.F == nodes[i - 1].desc.Fo, at + "widths do not chain (F must be the width of H[i-1])");
    if (d.variant == AGCN_VARIANT_SGC_LL) {
      AGCN_REQUIRE(nd.src == -1, at + "an SGC_LL layer takes no src (-1)");
      continue;
    }
    AGCN_REQUIRE(param_offsets[5 * (size_t)i + 4] >= 0, at + "a Reslap layer needs a beta offset");
    AGCN_REQUIRE(nd.src >= -1 && nd.src < i, at + "src must be an earlier node or -1");
    if (nd.src >= 0) {
      AGCN_REQUIRE(is_reslap(nodes[nd.src]), at + "a Reslap src must be a Reslap node (its L_all is this layer's L_prev)");
      AGCN_REQUIRE(lall_user[nd.src] < 0, at + "two Reslap layers name the same src (the L_all chain is linear)");
      lall_user[nd.src] = i;
    }
  }
  agcn_stack* s = new agcn_stack();
  s->nodes.assign(nodes, nodes + n_nodes);
  for (agcn_stack_node& nd : s->nodes) {
    // as functional._SGCLLFunction runs the layer classes
    nd.desc.flags = AGCN_SAVE_FOR_BACKWARD | (is_reslap(nd) ? AGCN_OUT_L_ALL : 0u);
    if (nd.kind == AGCN_NODE_SGCLL && !is_reslap(nd)) nd.src = -1;
  }
  s->Fm = Fm; s->Nt = Nt; s->loss_kind = loss_kind;
  s->off.assign(param_offsets, param_offsets + 5 * (size_t)n_nodes + 4);
  s->lall_user = lall_user;
  s->res_user = res_user;
  // prediction slots: H[i] is last read by node i+1 (the head for the last node) or by the BlockEnd it feeds x_res to;
  // L_all[i] by the Reslap layer it is L_prev of
  std::vector<int32_t> last_h(n_nodes), last_l(n_nodes);
  std::vector<bool> all(n_nodes, true), reslap(n_nodes);
  for (int i = 0; i < n_nodes; ++i) {
    last_h[i] = std::max(i + 1, res_user[i]);
    last_l[i] = std::max(i, lall_user[i]);
    reslap[i] = is_reslap(s->nodes[i]);
  }
  s->n_pred_h = assign_slots(last_h, all, &s->pred_h);
  s->n_pred_l = assign_slots(last_l, reslap, &s->pred_l);
  *out = s;
  return AGCN_OK;
}

int agcn_stack_create(const agcn_sgcll_desc* layer_descs, int32_t n_layers, int32_t Fm, int32_t Nt, int32_t loss_kind,
                      const int64_t* param_offsets, agcn_stack** out) {
  AGCN_REQUIRE(layer_descs && n_layers >= 1 && param_offsets && out, "stack_create: bad arguments");
  std::vector<agcn_stack_node> nodes(n_layers);
  for (int l = 0; l < n_layers; ++l) {
    AGCN_REQUIRE(layer_descs[l].variant == AGCN_VARIANT_SGC_LL, "stack_create: SGC_LL layers only (basic_AGCN.py:35-47)");
    AGCN_REQUIRE(l == 0 || layer_descs[l].F == layer_descs[l - 1].Fo, "stack_create: layer widths do not chain");
    nodes[l].kind = AGCN_NODE_SGCLL;
    nodes[l].desc = layer_descs[l];
    nodes[l].src = -1;
  }
  return agcn_stack_create_nodes(nodes.data(), n_layers, Fm, Nt, loss_kind, param_offsets, out);
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
  cudaStream_t st = (cudaStream_t)stream;
  const int nl = (int)s->nodes.size();
  const int32_t R = (int32_t)plan->R;
  auto P = [&](int l, int k) { return node_param(s, d_params, l, k); };
  auto G = [&](int l, int k) { return node_param(s, d_grads, l, k); };
  const int64_t* ho = &s->off[5 * (size_t)nl];
  if ((rc = forward_nodes(s, plan, w, d_X, d_Lint, d_params, true, stream))) return rc;
  // ---- DenseMol + GraphGatherMol + logits + loss, with every gradient of that part
  // (or the per-node head: logits + loss of every node)
  const agcn_sgcll_desc& last = s->nodes[nl - 1].desc;
  if (node_head(s))
    rc = agcn_node_head_loss_grad(plan, w.H[nl - 1], d_params + ho[2], d_params + ho[3], d_targets, d_weights, scale,
                                  last.Fo, s->Nt, d_loss, w.dA, d_grads + ho[2], d_grads + ho[3], w.head_work,
                                  w.head_work_bytes, stream);
  else
    rc = agcn_head_loss_grad_ex(plan, w.H[nl - 1], d_params + ho[0], d_params + ho[1], d_params + ho[2],
                                d_params + ho[3], d_targets, d_weights, scale, s->loss_kind, last.Fo, s->Fm, s->Nt,
                                d_loss, w.dA, d_grads + ho[0], d_grads + ho[1], d_grads + ho[2], d_grads + ho[3],
                                w.head_work, w.head_work_bytes, stream);
  if (rc) return rc;
  if (notify) notify(notify_user, nl, stream);
  // ---- backward, last node first; the first layer's input has no gradient unless the metric is differentiable.
  // dH[i-1] is written by node i (an SGC-LL layer's dX, or a BlockEnd's dpre, which is the gradient of its residual
  // add); a BlockEnd whose x_res is H[i-1] then adds dpre W^T to it, as autograd sums the two contributions.
  float* dcur = w.dA;
  for (int l = nl - 1; l >= 0; --l) {
    const agcn_stack_node& nd = s->nodes[l];
    const agcn_sgcll_desc& d = nd.desc;
    float* dnext = dcur == w.dA ? w.dB : w.dA;
    float* dprev = nullptr;   // dH[l-1]
    if (nd.kind == AGCN_NODE_BLOCK_END) {
      const long long n = (long long)R * d.Fo;
      act_grad_kernel<<<(unsigned)std::min<long long>((n + 255) / 256, 148 * 8), 256, 0, st>>>(
          dcur, w.H[l], w.dpre[l], n, d.activation == AGCN_ACT_RELU);
      AGCN_LAUNCH_CHECK();
      // dW = H[src]^T dpre, on the kernel functional._NodeLinear picks for this shape
      const int use_tc = (d.F <= 128 && d.F % 4 == 0 && d.Fo % 4 == 0 && R >= 32) ? 1 : 0;
      rc = agcn_gemm_tn(w.H[nd.src], nullptr, w.dpre[l], G(l, 0), R, d.F, d.Fo, 1, w.layer_work, use_tc, stream);
      if (rc) return rc;
      dprev = w.dpre[l];
      if (s->res_user[l - 1] >= 0) {   // more is added to dH[l-1]: keep dpre itself for this BlockEnd's dX product
        AGCN_CUDA(cudaMemcpyAsync(dnext, dprev, (size_t)R * d.Fo * sizeof(float), cudaMemcpyDeviceToDevice, st));
        dprev = dnext;
      }
    } else {
      const bool full = d.laplacian_mode == AGCN_LAP_PAPER && d.metric_grad == AGCN_METRIC_GRAD_FULL;
      const bool reslap = is_reslap(nd);
      const float* Lprev = (reslap && nd.src >= 0) ? w.Lall[nd.src] : nullptr;
      dprev = (l > 0 || full) ? dnext : nullptr;
      rc = agcn_sgcll_backward(&d, plan, l == 0 ? d_X : w.H[l - 1], d_Lint, Lprev, P(l, 2), P(l, 0), P(l, 3), P(l, 4),
                               w.H[l], dcur, reslap ? w.dLall[l] : nullptr, w.saved[l], dprev, G(l, 2), G(l, 0),
                               G(l, 1), G(l, 3), G(l, 4), Lprev ? w.dLall[nd.src] : nullptr, w.layer_work,
                               w.layer_work_bytes, stream);
      if (rc) return rc;
    }
    if (notify) notify(notify_user, l, stream);
    if (l > 0 && s->res_user[l - 1] >= 0) {   // BlockEnd b's x_res is H[l-1]: dH[l-1] += dpre_b W_b^T
      const int bn = s->res_user[l - 1];
      const agcn_sgcll_desc& bd = s->nodes[bn].desc;
      rc = agcn_node_gemm(w.dpre[bn], bd.Fo, P(bn, 0), bd.Fo, 1, dprev, bd.F, R, bd.F, bd.Fo, nullptr, nullptr, 1,
                          AGCN_ACT_LINEAR, w.layer_work, stream);
      if (rc) return rc;
    }
    dcur = dprev;
  }
  return AGCN_OK;
}

int agcn_stack_predict_workspace_bytes(const agcn_stack* s, const agcn_plan* plan, size_t* bytes) {
  AGCN_REQUIRE(s && plan && bytes, "stack_predict_workspace_bytes: null pointer");
  StackWork w;
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
  StackWork w;
  int rc = carve_predict(s, plan, d_work, &w);
  if (rc) return rc;
  if (w.bytes > work_bytes) {
    set_error("stack_predict: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  if ((rc = forward_nodes(s, plan, w, d_X, d_Lint, d_params, false, stream))) return rc;
  const int nl = (int)s->nodes.size();
  const int64_t* ho = &s->off[5 * (size_t)nl];
  const int32_t Fh = s->nodes.back().desc.Fo;
  if (node_head(s))
    return agcn_node_head_predict(plan, w.H[nl - 1], d_params + ho[2], d_params + ho[3], d_targets, d_weights, scale, Fh,
                                  s->Nt, d_probs, d_loss, w.head_work, w.head_work_bytes, stream);
  return agcn_head_predict(plan, w.H[nl - 1], d_params + ho[0], d_params + ho[1], d_params + ho[2], d_params + ho[3],
                           d_targets, d_weights, scale, s->loss_kind, Fh, s->Fm, s->Nt, d_probs, d_loss, w.head_work,
                           w.head_work_bytes, stream);
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
