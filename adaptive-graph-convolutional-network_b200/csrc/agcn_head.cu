// The layers that follow the last SGC-LL layer in the reference's networks (basic_AGCN.py:35-47), as ONE
// loss-and-gradient call on the packed layout (SURVEY.md section 8f, rows 1 and 3):
//
//   DenseMol        h_i W_d + b_d, no activation                 models/layers/dense_layer.py:33-50
//   GraphGatherMol  per-graph sum over the real atoms, tanh      models/layers/graphgather.py:50-78
//   logits          n_tasks independent [n_feature, 2] heads     models/operators/model_operatos.py:792-864
//   loss            weighted sigmoid cross-entropy / batch size  models/tf_modules/multitask_classifier.py:41-44,187-209
//   or, for regression, n_tasks [n_feature, 1] heads and the weighted L2 / batch size of DeepChem's
//   MultitaskGraphRegressor (models/tf_modules/multitask_regressor.py, final_loss='weighted_L2'; parity unpinned)
//
// DenseMol is linear, so the gather commutes with it: sum_i (h_i W + b) = (sum_i h_i) W + n_g b.  The dense GEMM
// then has B rows instead of R = sum n_g.  The n_tasks heads are one [n_feature, 2 n_tasks] matrix.  Every
// contraction runs on the tcgen05 3xTF32 GEMMs of agcn_tc_gemm.cu; the cross-entropy (or the weighted L2) and its
// gradient are the epilogue of the logits GEMM, so the [B, 2 n_tasks] logits never reach HBM as logits.
#include <algorithm>

#include "agcn_internal.cuh"

namespace agcn {

// hsum[g, :] = sum of the rows of graph g          (one warp per graph; every row load of the warp is in flight at
// once: lanes walk the graph's rows as one contiguous [n_g * F] range, fixed summation order per column)
__global__ void segment_sum_kernel(const float* __restrict__ H, const int32_t* __restrict__ node_off, int B, int F,
                                   float* __restrict__ hsum) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (g >= B) return;
  const int r0 = node_off[g], r1 = node_off[g + 1];
  if (F % 32 == 0) {
    // lane owns columns lane, lane + 32, ...: consecutive lanes read consecutive addresses of every row
    for (int c = lane; c < F; c += 32) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      int r = r0;
      for (; r + 4 <= r1; r += 4) {
        s0 += __ldg(H + (int64_t)r * F + c);
        s1 += __ldg(H + (int64_t)(r + 1) * F + c);
        s2 += __ldg(H + (int64_t)(r + 2) * F + c);
        s3 += __ldg(H + (int64_t)(r + 3) * F + c);
      }
      for (; r < r1; ++r) s0 += __ldg(H + (int64_t)r * F + c);
      hsum[(int64_t)g * F + c] = (s0 + s1) + (s2 + s3);
    }
    return;
  }
  for (int c = lane; c < F; c += 32) {
    float s = 0.f;
    for (int r = r0; r < r1; ++r) s += H[(int64_t)r * F + c];
    hsum[(int64_t)g * F + c] = s;
  }
}

// Labels as the reference feeds them (multitask_classifier.py:147-152,171-185: one label and one weight per sample and
// task; the one-hot encoding happens inside the graph, :196-199 tf.one_hot(label, 2)) -> the [B, 2 T] targets / per-logit
// weights the loss epilogue reads.  Plain loads of the inputs: pinned host arrays are read in place over PCIe (4 bytes of
// label + weight per task instead of 16 bytes of expanded rows); a few persistent CTAs so that the kernel can live beside
// the previous training step like the pack kernels.
__global__ void __launch_bounds__(1024) expand_labels_kernel(const uint8_t* __restrict__ y, const float* __restrict__ w,
                                                             long long n, float2* __restrict__ targets,
                                                             float2* __restrict__ weights) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const float yv = y[e] ? 1.f : 0.f, wv = w[e];
    targets[e] = make_float2(1.f - yv, yv);
    weights[e] = make_float2(wv, wv);
  }
}

// mol = tanh(a), a = pre + n_g b   (graphgather.py:77); `pre` is overwritten with tanh'(a) = sech^2(a) evaluated as
// 4 e / (1 + e)^2, e = exp(-2 |a|): the sum over a molecule's atoms saturates the tanh, and 1 - mol^2 would then
// cancel to a handful of significant bits (errors of 1e-4 .. 1e-3 relative in every gradient behind it)
__global__ void gather_tanh_kernel(float* __restrict__ pre, const float* __restrict__ b,
                                   const int32_t* __restrict__ n_nodes, int B, int Fm, float* __restrict__ mol) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)B * Fm) return;
  const int g = (int)(e / Fm), c = (int)(e % Fm);
  const float a = pre[e] + (float)n_nodes[g] * b[c];
  mol[e] = tanhf(a);
  const float ex = expf(-2.f * fabsf(a));
  pre[e] = 4.f * ex / ((1.f + ex) * (1.f + ex));
}

// dpre = dmol tanh'(a), in place over dmol
__global__ void tanh_bwd_kernel(const float* __restrict__ dtanh, float* __restrict__ dmol, int64_t total) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  dmol[e] = dmol[e] * dtanh[e];
}

// out[c] = sum_r w_r M[r, c]  (w == NULL: plain column sums): 32 columns per CTA, rows over 8 warps, fixed order
__global__ void __launch_bounds__(256) weighted_colsum_kernel(const float* __restrict__ M, int ld, int rows, int cols,
                                                              const int32_t* __restrict__ w, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < cols)
    for (int r = wid; r < rows; r += 8) s += (w ? (float)w[r] : 1.f) * M[(int64_t)r * ld + c];
  red[wid][lane] = s;
  __syncthreads();
  if (wid == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][lane];
    out[c] = t;
  }
}

// dH[r, :] = dhsum[graph(r), :]      (one warp per graph)
__global__ void segment_broadcast_kernel(const float* __restrict__ dhsum, const int32_t* __restrict__ node_off, int B,
                                         int F, float* __restrict__ dH) {
  const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (g >= B) return;
  const int r0 = node_off[g], r1 = node_off[g + 1];
  for (int c = lane; c < F; c += 32) {
    const float v = dhsum[(int64_t)g * F + c];
    for (int r = r0; r < r1; ++r) dH[(int64_t)r * F + c] = v;
  }
}

// dst[r, 0:cols] = src[r, 0:cols]  (different row pitches)
__global__ void copy_pitched_kernel(const float* __restrict__ src, int lds, float* __restrict__ dst, int ldd, int rows,
                                    int cols) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)rows * cols) return;
  const int r = (int)(e / cols), c = (int)(e % cols);
  dst[(int64_t)r * ldd + c] = src[(int64_t)r * lds + c];
}

// Single-task multi-class head (SingletaskGraphClassifier: models/tf_modules/singletask_classifier.py:124-151 with
// get_loss_fn('softmax_cross_entropy'), multitask_classifier.py:45-48): one warp per sample,
//   loss_b = w_b * sum_c y_c (logsumexp(x) - x_c),   d loss / d x_c = w_b (softmax_c * sum y - y_c) * scale
// GRAD (training): `logits` [B, ld] is overwritten by the gradient.  Otherwise (prediction) probs[b, :] = softmax(x_b)
// = exp(x_b - logsumexp(x_b)), and y may be NULL.  With y, part[b] receives loss_b * scale: one expression for both
// calls, so the evaluation loss is bit-identical to the training loss.
template <bool GRAD>
__global__ void softmax_ce_kernel(float* __restrict__ logits, int ld, const float* __restrict__ y,
                                  const float* __restrict__ w, int B, int C, float scale, float* __restrict__ probs,
                                  float* __restrict__ part) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  float* x = logits + (int64_t)b * ld;
  const float* yb = y ? y + (int64_t)b * C : nullptr;
  float mx = -INFINITY;
  for (int c = lane; c < C; c += 32) mx = fmaxf(mx, x[c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float se = 0.f, sy = 0.f, sxy = 0.f;
  for (int c = lane; c < C; c += 32) {
    se += expf(x[c] - mx);
    if (GRAD || yb) {
      sy += yb[c];
      sxy += yb[c] * x[c];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, o);
    sy += __shfl_xor_sync(0xffffffffu, sy, o);
    sxy += __shfl_xor_sync(0xffffffffu, sxy, o);
  }
  const float lse = mx + logf(se);
  if (GRAD) {
    const float wb = w[b];
    for (int c = lane; c < C; c += 32) x[c] = wb * (expf(x[c] - lse) * sy - yb[c]) * scale;
  } else {
    float* pb = probs + (int64_t)b * C;
    for (int c = lane; c < C; c += 32) pb[c] = expf(x[c] - lse);
  }
  if (yb && lane == 0) part[b] = w[b] * (lse * sy - sxy) * scale;
}

__global__ void sum_parts_kernel(const float* __restrict__ parts, int n, float* __restrict__ out) {
  __shared__ float red[256];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += parts[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = red[0];
}

namespace {

// contraction over the rows: tensor cores when the shape allows it (>= 32 rows, TMA-compatible), CUDA cores otherwise
int tn_any(const GemmTNArgs& t, cudaStream_t st) {
  if (tc_gemm_tn_supported(t)) return tc_gemm_tn(t, st);
  return gemm_tn(t, st);
}
size_t tn_any_partial(const GemmTNArgs& t) {
  return std::max(tc_gemm_tn_partial_floats(t), gemm_tn_partial_floats(t.M, t.Kd, t.N, t.S));
}

inline int pad4(int x) { return (x + 3) & ~3; }

// The forward areas come first: they are agcn_head_predict's whole work area, and training adds its backward areas
// behind them.
struct HeadWork {
  float *hsum, *pre, *mol, *dlog, *loss_part, *tcB;
  float *dmol, *dhsum, *dWh_pad, *tcC, *tcD, *tn_part, *splitk;
  size_t bytes;
};

HeadWork carve_head(const agcn_plan* plan, int Fh, int Fm, int Nt, bool train, void* base) {
  Arena c(base);
  const size_t B = plan->B;
  const int Ntp = pad4(Nt);
  HeadWork w{};
  w.hsum = c.take(B * Fh);
  w.pre = c.take(B * Fm);
  w.mol = c.take(B * Fm);
  w.dlog = c.take(B * Ntp);   // row pitch Ntp: d loss / d logits (pad columns stay zero), or the single-task logits
  GemmArgs g;
  g.M = (int)B; g.N = Nt; g.Z = 1; g.prob = 1;  // sized for the tiles of the fused-loss product
  w.loss_part = c.take(std::max((size_t)tc_gemm_loss_parts(g), B) + 64);
  w.tcB = c.take(tc_gemm_scratch_floats(Nt, Fm, 1, 1));   // head_W             (logits = mol head_W)
  if (train) {
    w.dmol = c.take(B * Fm);
    w.dhsum = c.take(B * Fh);
    w.dWh_pad = c.take((size_t)Fm * Ntp);
    w.tcC = c.take(tc_gemm_scratch_floats(Fm, Nt, 1, 1));   // head_W^T operand   (dmol  = dlog head_W^T)
    w.tcD = c.take(tc_gemm_scratch_floats(Fh, Fm, 1, 1));   // dense_W^T operand  (dhsum = dpre dense_W^T)
    GemmTNArgs t;
    t.M = (int)B; t.Kd = std::min(Fm, 128); t.N = Ntp; t.S = 1;
    size_t tn = tn_any_partial(t);
    t.Kd = Fh; t.N = Fm;
    tn = std::max(tn, tn_any_partial(t));
    w.tn_part = c.take(tn);
    w.splitk = c.take((size_t)8 * B * std::max(Fm, Fh));  // split-K partial sums of the two long contractions
  }
  w.bytes = c.bytes;
  return w;
}

// Parameter gradients of agcn_head_loss_grad_ex
struct HeadGrads {
  float *dH, *ddense_W, *ddense_b, *dhead_W, *dhead_b;
};

// Both head calls.  The forward runs the same products with the same tile configurations for training (grads set) and
// prediction (grads NULL): `pre` on the CUDA cores, the logits on the tensor cores with the loss (or the probabilities)
// in their epilogue, the single-task softmax in softmax_ce_kernel.  The evaluation loss is therefore bit-identical to
// the training loss.  Prediction writes the probabilities (weighted L2: the values) to d_probs and the loss to d_loss
// when targets are given; training writes the loss and every gradient.
int head_run(const char* who, const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
             const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights, float scale,
             int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_probs, float* d_loss, const HeadGrads* gr,
             void* d_work, size_t work_bytes, cudaStream_t st) {
  const std::string at = std::string(who) + ": ";
  AGCN_REQUIRE(loss_kind == AGCN_LOSS_SIGMOID_CE || loss_kind == AGCN_LOSS_SOFTMAX_CE ||
                   loss_kind == AGCN_LOSS_WEIGHTED_L2,
               at + "unknown loss_kind");
  // the logits GEMM carries the loss epilogue on the tensor cores: its contraction (Fm) must reach one k-block with
  // 16-byte operand pitches; every other contraction falls back to the CUDA-core kernels when its shape is not
  // TMA-compatible (e.g. 12 tasks: Nt = 24)
  AGCN_REQUIRE(Fh >= 1 && Fm >= 32 && Fm % 4 == 0 && Nt >= 1,
               at + "unsupported sizes (need Fm >= 32 and a multiple of 4)");
  const bool train = gr != nullptr, softmax = loss_kind == AGCN_LOSS_SOFTMAX_CE;
  AGCN_REQUIRE(train || loss_kind != AGCN_LOSS_SIGMOID_CE || Nt % 2 == 0,
               at + "the multitask head needs two logits per task (Nt even)");
  int rc = plan_use(plan, st);
  if (rc) return rc;
  HeadWork w = carve_head(plan, Fh, Fm, Nt, train, d_work);
  if (w.bytes > work_bytes) {
    set_error(at + "workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  const int B = plan->B, Ntp = pad4(Nt);
  cudaStream_t side = plan->side;

  GemmArgs g_pre, g_log;
  g_pre.M = B; g_pre.N = Fm; g_pre.Kd = Fh;
  g_pre.A0 = w.hsum; g_pre.lda0 = Fh;
  g_pre.B = d_dense_W; g_pre.ldb = Fm;
  g_pre.C = w.pre; g_pre.ldc = Fm;
  g_log.M = B; g_log.N = Nt; g_log.Kd = Fm;
  g_log.A0 = w.mol; g_log.lda0 = Fm;
  g_log.B = d_head_W; g_log.ldb = Nt;
  g_log.C = w.dlog; g_log.ldc = Ntp;
  g_log.bias = d_head_b;
  if (!softmax) {  // sigmoid cross-entropy or weighted L2: the loss is the GEMM's epilogue
    g_log.l2 = loss_kind == AGCN_LOSS_WEIGHTED_L2;
    if (d_targets) {
      g_log.bce_y = d_targets; g_log.bce_w = d_weights; g_log.bce_ld = Nt; g_log.bce_scale = scale;
      g_log.loss_part = w.loss_part;
    }
    if (!train) {  // C receives the pairwise softmax of the logits (weighted L2: the values x) instead of the gradient
      g_log.C = d_probs; g_log.ldc = Nt;
      g_log.prob = 1;
    }
  }
  AGCN_REQUIRE(tc_gemm_supported(g_log), at + "operands are not TMA-compatible (alignment)");
  GemmArgs g_dmol, g_dhs;
  g_dmol.M = B; g_dmol.N = Fm; g_dmol.Kd = Nt;
  g_dmol.A0 = w.dlog; g_dmol.lda0 = Ntp;
  g_dmol.B = d_head_W; g_dmol.ldb = Nt; g_dmol.transB = 1;  // head_W is [Fm, Nt] = [N, Kd]
  g_dmol.C = w.dmol; g_dmol.ldc = Fm; g_dmol.split_k_partial = w.splitk;
  g_dhs.M = B; g_dhs.N = Fh; g_dhs.Kd = Fm;
  g_dhs.A0 = w.dmol; g_dhs.lda0 = Fm;
  g_dhs.B = d_dense_W; g_dhs.ldb = Fm; g_dhs.transB = 1;    // dense_W is [Fh, Fm] = [N, Kd]
  g_dhs.C = w.dhsum; g_dhs.ldc = Fh; g_dhs.split_k_partial = w.splitk;
  // dhsum = dpre dense_W^T is [B, Fm] x [Fm, Fh] with Fh = 64: eight 128-row tiles of eight k-blocks each -- a latency chain
  // of 30 us on 8 SMs on the tensor-core kernel, 12 us spread over every SM on the CUDA cores (33 MFLOP)
  const bool tc_dmol = train && tc_gemm_supported(g_dmol),
             tc_dhs = train && tc_gemm_supported(g_dhs) && (int64_t)B * Fh * Fm > (1ll << 26);

  // parameter operands (hi / lo split, K-major) on the side stream while the gather runs
  AGCN_CUDA(cudaEventRecord(plan->ev_side_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(side, plan->ev_side_fork, 0));
  if ((rc = tc_gemm_split_b(g_log, w.tcB, side))) return rc;
  if (tc_dmol && (rc = tc_gemm_split_b(g_dmol, w.tcC, side))) return rc;
  if (tc_dhs && (rc = tc_gemm_split_b(g_dhs, w.tcD, side))) return rc;
  if (train && (rc = zero_async(w.dlog, (size_t)B * Ntp, side))) return rc;  // pad columns of dlog
  AGCN_CUDA(cudaEventRecord(plan->ev_side_join, side));

  // GraphGatherMol + DenseMol (commuted) + tanh.  `pre` feeds a tanh that the sum over a molecule's atoms saturates:
  // tanh'(a) = sech^2(a) has relative sensitivity 2 |da|, so the absolute error of this [B, Fh] x [Fh, Fm] product (a
  // few MFLOP) decides the accuracy of every gradient behind it.  Plain fp32 FMAs (gemm_rows) keep it at fp32 rounding
  // level; 3xTF32 is ~4x coarser.
  segment_sum_kernel<<<(B + 7) / 8, 256, 0, st>>>(d_H, plan->d_node_off, B, Fh, w.hsum);
  AGCN_LAUNCH_CHECK();
  if ((rc = gemm_rows(g_pre, st))) return rc;
  {
    const int64_t total = (int64_t)B * Fm;
    gather_tanh_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w.pre, d_dense_b, plan->d_n, B, Fm, w.mol);
    AGCN_LAUNCH_CHECK();
  }
  // logits + loss epilogue: C receives d loss / d logits (training), the probabilities (prediction) or, for the
  // single-task head, the logits; the loss its per-warp partial sums
  AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));
  if ((rc = tc_gemm(g_log, w.tcB, st))) return rc;
  int n_parts = tc_gemm_loss_parts(g_log);
  if (softmax) {  // softmax cross-entropy row by row
    (train ? softmax_ce_kernel<true> : softmax_ce_kernel<false>)<<<(B + 7) / 8, 256, 0, st>>>(
        w.dlog, Ntp, d_targets, d_weights, B, Nt, scale, d_probs, w.loss_part);
    AGCN_LAUNCH_CHECK();
    n_parts = B;
  }
  if (d_loss) {
    sum_parts_kernel<<<1, 256, 0, st>>>(w.loss_part, n_parts, d_loss);
    AGCN_LAUNCH_CHECK();
  }
  if (!train) return AGCN_OK;

  // parameter gradients of the heads on the side stream, beside the chain back to dH
  AGCN_CUDA(cudaEventRecord(plan->ev_side_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(side, plan->ev_side_fork, 0));
  weighted_colsum_kernel<<<(Nt + 31) / 32, 256, 0, side>>>(w.dlog, Ntp, B, Nt, nullptr, gr->dhead_b);
  AGCN_LAUNCH_CHECK();
  for (int f0 = 0; f0 < Fm; f0 += 128) {  // dhead_W = mol^T dlog, 128 rows of the result per contraction
    GemmTNArgs t;
    t.M = B; t.Kd = std::min(128, Fm - f0); t.N = Ntp; t.S = 1;
    t.A0 = w.mol + f0; t.lda0 = Fm;
    t.D = w.dlog; t.ldd = Ntp;
    t.out = w.dWh_pad + (size_t)f0 * Ntp; t.partial = w.tn_part;
    if ((rc = tn_any(t, side))) return rc;
  }
  {
    const int64_t total = (int64_t)Fm * Nt;
    copy_pitched_kernel<<<(unsigned)((total + 255) / 256), 256, 0, side>>>(w.dWh_pad, Ntp, gr->dhead_W, Nt, Fm, Nt);
    AGCN_LAUNCH_CHECK();
  }

  // main stream: dmol = dlog head_W^T, through tanh, ddense_b, dhsum, dH
  auto gemm_any = [&](const GemmArgs& g, const float* scratch, bool tc) { return tc ? tc_gemm(g, scratch, st) : gemm_rows(g, st); };
  if ((rc = gemm_any(g_dmol, w.tcC, tc_dmol))) return rc;
  {
    const int64_t total = (int64_t)B * Fm;
    tanh_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w.pre, w.dmol, total);  // dmol := dpre
    AGCN_LAUNCH_CHECK();
  }
  if ((rc = gemm_any(g_dhs, w.tcD, tc_dhs))) return rc;
  segment_broadcast_kernel<<<(B + 7) / 8, 256, 0, st>>>(w.dhsum, plan->d_node_off, B, Fh, gr->dH);
  AGCN_LAUNCH_CHECK();
  // dense parameter gradients (need dpre; the dhead_W contraction on the side stream is done with tn_part by now
  // only if we wait for it, so they follow it on the side stream)
  AGCN_CUDA(cudaEventRecord(plan->ev_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(side, plan->ev_fork, 0));
  weighted_colsum_kernel<<<(Fm + 31) / 32, 256, 0, side>>>(w.dmol, Fm, B, Fm, plan->d_n, gr->ddense_b);
  AGCN_LAUNCH_CHECK();
  {
    GemmTNArgs t;  // ddense_W = hsum^T dpre
    t.M = B; t.Kd = Fh; t.N = Fm; t.S = 1;
    t.A0 = w.hsum; t.lda0 = Fh;
    t.D = w.dmol; t.ldd = Fm;
    t.out = gr->ddense_W; t.partial = w.tn_part;
    if ((rc = tn_any(t, side))) return rc;
  }
  AGCN_CUDA(cudaEventRecord(plan->ev_side_join, side));
  AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));
  return AGCN_OK;
}

}  // namespace
}  // namespace agcn

using namespace agcn;

extern "C" {

int agcn_expand_labels(const uint8_t* y, const float* w, int32_t B, int32_t n_tasks, float* d_targets, float* d_weights,
                       void* stream) {
  AGCN_REQUIRE(y && w && d_targets && d_weights && B >= 1 && n_tasks >= 1, "expand_labels: bad arguments");
  AGCN_REQUIRE((reinterpret_cast<uintptr_t>(d_targets) & 7) == 0 && (reinterpret_cast<uintptr_t>(d_weights) & 7) == 0,
               "expand_labels: outputs must be 8-byte aligned");
  const long long n = (long long)B * n_tasks;
  const unsigned grid = (unsigned)std::max<long long>(1, std::min<long long>((n + 1023) / 1024, 8));
  expand_labels_kernel<<<grid, 1024, 0, (cudaStream_t)stream>>>(y, w, n, reinterpret_cast<float2*>(d_targets),
                                                               reinterpret_cast<float2*>(d_weights));
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

int agcn_head_workspace_bytes(const agcn_plan* plan, int32_t Fh, int32_t Fm, int32_t Nt, size_t* bytes) {
  AGCN_REQUIRE(plan && bytes && Fh >= 1 && Fm >= 1 && Nt >= 1, "head_workspace_bytes: bad arguments");
  *bytes = carve_head(plan, Fh, Fm, Nt, true, nullptr).bytes + 256;
  return AGCN_OK;
}

int agcn_head_loss_grad(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                        const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                        float scale, int32_t Fh, int32_t Fm, int32_t Nt, float* d_loss, float* d_dH,
                        float* d_ddense_W, float* d_ddense_b, float* d_dhead_W, float* d_dhead_b, void* d_work,
                        size_t work_bytes, void* stream) {
  return agcn_head_loss_grad_ex(plan, d_H, d_dense_W, d_dense_b, d_head_W, d_head_b, d_targets, d_weights, scale,
                                AGCN_LOSS_SIGMOID_CE, Fh, Fm, Nt, d_loss, d_dH, d_ddense_W, d_ddense_b, d_dhead_W,
                                d_dhead_b, d_work, work_bytes, stream);
}

int agcn_head_loss_grad_ex(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                           const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                           float scale, int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_loss,
                           float* d_dH, float* d_ddense_W, float* d_ddense_b, float* d_dhead_W, float* d_dhead_b,
                           void* d_work, size_t work_bytes, void* stream) {
  AGCN_REQUIRE(plan && d_H && d_dense_W && d_dense_b && d_head_W && d_head_b && d_targets && d_weights && d_loss &&
                   d_dH && d_ddense_W && d_ddense_b && d_dhead_W && d_dhead_b && d_work,
               "head_loss_grad: null pointer");
  const HeadGrads gr{d_dH, d_ddense_W, d_ddense_b, d_dhead_W, d_dhead_b};
  return head_run("head_loss_grad", plan, d_H, d_dense_W, d_dense_b, d_head_W, d_head_b, d_targets, d_weights, scale,
                  loss_kind, Fh, Fm, Nt, nullptr, d_loss, &gr, d_work, work_bytes, (cudaStream_t)stream);
}

int agcn_head_predict_workspace_bytes(const agcn_plan* plan, int32_t Fh, int32_t Fm, int32_t Nt, size_t* bytes) {
  AGCN_REQUIRE(plan && bytes && Fh >= 1 && Fm >= 1 && Nt >= 1, "head_predict_workspace_bytes: bad arguments");
  *bytes = carve_head(plan, Fh, Fm, Nt, false, nullptr).bytes + 256;
  return AGCN_OK;
}

int agcn_head_predict(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                      const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                      float scale, int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_probs, float* d_loss,
                      void* d_work, size_t work_bytes, void* stream) {
  AGCN_REQUIRE(!d_targets == !d_weights && !d_targets == !d_loss,
               "head_predict: d_targets, d_weights and d_loss must be all NULL or all set");
  AGCN_REQUIRE(plan && d_H && d_dense_W && d_dense_b && d_head_W && d_head_b && d_probs && d_work,
               "head_predict: null pointer");
  return head_run("head_predict", plan, d_H, d_dense_W, d_dense_b, d_head_W, d_head_b, d_targets, d_weights, scale,
                  loss_kind, Fh, Fm, Nt, d_probs, d_loss, nullptr, d_work, work_bytes, (cudaStream_t)stream);
}

}  // extern "C"
