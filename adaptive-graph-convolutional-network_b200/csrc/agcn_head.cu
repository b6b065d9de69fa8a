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
//
// The per-node head (agcn_node_head_*, the part labels of the reference's segmentation network; restated, parity
// unpinned) has no DenseMol, gather or tanh: logits H head_W + head_b for every packed row, then the single-task head's
// row softmax over R rows instead of B.
#include <algorithm>

#include "agcn_internal.cuh"

namespace agcn {

constexpr int HEAD_GRAPHS = 4;  // graphs per CTA of head_fwd_kernel / head_bwd_kernel (B = 1024: 256 CTAs)

// GraphGatherMol + DenseMol (commuted) + tanh for HEAD_GRAPHS graphs x 256 columns of Fm:
//   hsum[g, :] = sum of the rows of graph g,  a = hsum[g, :] dense_W + n_g dense_b,  mol = tanh(a),
//   dtanh = tanh'(a) = sech^2(a) evaluated as 4 e / (1 + e)^2, e = exp(-2 |a|): the sum over a molecule's atoms
//   saturates the tanh, and 1 - mol^2 would then cancel to a handful of significant bits (errors of 1e-4 .. 1e-3
//   relative in every gradient behind it).
// The row sums run 64 columns of Fh at a time, one thread per (graph, column); for Fh % 32 == 0 each thread keeps four
// partial sums over rows r0 + 4i + j (eight rows in flight), the rest go to the first, and the result is
// (s0 + s1) + (s2 + s3).  The product runs one thread per column in fp32, four k at a time with the expression of
// gemm_rows_kernel (groups aligned to k = 0, zero past Fh), so `pre` is what gemm_rows computes.  Every CTA sums its
// graphs' rows; those of blockIdx.y == 0 write hsum (ddense_W = hsum^T dpre reads it).
__global__ void __launch_bounds__(256) head_fwd_kernel(const float* __restrict__ H, const int32_t* __restrict__ node_off,
                                                       const int32_t* __restrict__ n_nodes,
                                                       const float* __restrict__ W, const float* __restrict__ b, int B,
                                                       int Fh, int Fm, float* __restrict__ hsum,
                                                       float* __restrict__ dtanh, float* __restrict__ mol) {
  __shared__ float hs[HEAD_GRAPHS][64];
  const int t = threadIdx.x, g0 = blockIdx.x * HEAD_GRAPHS, c = blockIdx.y * 256 + t;
  const int sg = t >> 6, sc = t & 63, g = g0 + sg;
  const int r0 = g < B ? node_off[g] : 0, r1 = g < B ? node_off[g + 1] : 0;
  float acc[HEAD_GRAPHS];
#pragma unroll
  for (int i = 0; i < HEAD_GRAPHS; ++i) acc[i] = 0.f;
  for (int k0 = 0; k0 < Fh; k0 += 64) {
    const int col = k0 + sc;
    float s = 0.f;
    if (col < Fh) {
      const float* __restrict__ h = H + col;
      if (Fh % 32 == 0) {
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int r = r0;
        for (; r + 8 <= r1; r += 8) {
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = __ldg(h + (int64_t)(r + j) * Fh);
          s0 += v[0]; s1 += v[1]; s2 += v[2]; s3 += v[3];
          s0 += v[4]; s1 += v[5]; s2 += v[6]; s3 += v[7];
        }
        if (r + 4 <= r1) {
          s0 += __ldg(h + (int64_t)r * Fh);
          s1 += __ldg(h + (int64_t)(r + 1) * Fh);
          s2 += __ldg(h + (int64_t)(r + 2) * Fh);
          s3 += __ldg(h + (int64_t)(r + 3) * Fh);
          r += 4;
        }
        for (; r < r1; ++r) s0 += __ldg(h + (int64_t)r * Fh);
        s = (s0 + s1) + (s2 + s3);
      } else {
        for (int r = r0; r < r1; ++r) s += __ldg(h + (int64_t)r * Fh);
      }
      if (g < B && blockIdx.y == 0) hsum[(int64_t)g * Fh + col] = s;
    }
    hs[sg][sc] = s;
    __syncthreads();
    if (c < Fm) {
      const int kn = min(64, Fh - k0);   // hs[.][k] == 0 for k >= kn
      const float* __restrict__ w = W + (int64_t)k0 * Fm + c;
      for (int k = 0; k < kn; k += 4) {
        const float b0 = __ldg(w + (int64_t)k * Fm);
        const float b1 = k + 1 < kn ? __ldg(w + (int64_t)(k + 1) * Fm) : 0.f;
        const float b2 = k + 2 < kn ? __ldg(w + (int64_t)(k + 2) * Fm) : 0.f;
        const float b3 = k + 3 < kn ? __ldg(w + (int64_t)(k + 3) * Fm) : 0.f;
#pragma unroll
        for (int i = 0; i < HEAD_GRAPHS; ++i)
          acc[i] += hs[i][k] * b0 + hs[i][k + 1] * b1 + hs[i][k + 2] * b2 + hs[i][k + 3] * b3;
      }
    }
    __syncthreads();
  }
  if (c >= Fm) return;
  const float bc = b[c];
#pragma unroll
  for (int i = 0; i < HEAD_GRAPHS; ++i) {
    if (g0 + i >= B) break;
    const int64_t e = (int64_t)(g0 + i) * Fm + c;
    const float a = acc[i] + (float)n_nodes[g0 + i] * bc;
    mol[e] = tanhf(a);
    const float ex = expf(-2.f * fabsf(a));
    dtanh[e] = 4.f * ex / ((1.f + ex) * (1.f + ex));
  }
}

// The way back from d loss / d mol to dH for HEAD_GRAPHS graphs per CTA (dynamic shared memory: HEAD_GRAPHS x (Fm + Fh)
// floats).  dmol arrives as `chunks` split-K partial sums chunk_stride floats apart (chunks == 1: dmol itself), added in
// the order of reduce_chunks_kernel; then
//   dpre = dmol tanh'(a)                       (written: ddense_W and ddense_b read it; dpre may alias dmol)
//   dhsum[g, j] = sum_c dpre[g, c] dense_W[j, c]: one thread per (graph, j), fp32, four c at a time with the expression
//                 of gemm_rows_kernel, so dhsum is what gemm_rows computes; dense_W passes through shared memory in
//                 64 x 32 tiles read along its rows
//   dH[r, :] = dhsum[g, :] for every row r of graph g
// dH == NULL: dpre only (the large shapes of head_run take dhsum from the tensor cores).
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* dmol, int64_t chunk_stride, int chunks,
                                                       const float* __restrict__ dtanh, const float* __restrict__ W,
                                                       const int32_t* __restrict__ node_off, int B, int Fh, int Fm,
                                                       float* dpre, float* __restrict__ dH) {
  extern __shared__ float sp[];  // [HEAD_GRAPHS][Fm] dpre, then [HEAD_GRAPHS][Fh] dhsum
  __shared__ float ws[64][33];   // dense_W[j0 + jj, c0 + cc]
  float* dh = sp + HEAD_GRAPHS * Fm;
  const int t = threadIdx.x, g0 = blockIdx.x * HEAD_GRAPHS, ng = min(HEAD_GRAPHS, B - g0);
  for (int c = t; c < Fm; c += 256) {
#pragma unroll
    for (int i = 0; i < HEAD_GRAPHS; ++i) {
      float v = 0.f;
      if (i < ng) {
        const int64_t e = (int64_t)(g0 + i) * Fm + c;
        float s = 0.f;
        for (int k = 0; k < chunks; ++k) s += dmol[k * chunk_stride + e];
        v = s * dtanh[e];
        dpre[e] = v;
      }
      sp[i * Fm + c] = v;
    }
  }
  if (!dH) return;
  const int i = t >> 6, jj = t & 63;   // 256 threads = HEAD_GRAPHS x 64
  const float* p = sp + i * Fm;
  for (int j0 = 0; j0 < Fh; j0 += 64) {
    float acc = 0.f;
    for (int c0 = 0; c0 < Fm; c0 += 32) {
      __syncthreads();
      for (int e = t; e < 64 * 32; e += 256) {
        const int r = e >> 5, cc = e & 31;
        ws[r][cc] = j0 + r < Fh && c0 + cc < Fm ? __ldg(W + (int64_t)(j0 + r) * Fm + c0 + cc) : 0.f;
      }
      __syncthreads();
      const int cn = min(32, Fm - c0);   // a multiple of 4
      for (int cc = 0; cc < cn; cc += 4)
        acc += p[c0 + cc] * ws[jj][cc] + p[c0 + cc + 1] * ws[jj][cc + 1] + p[c0 + cc + 2] * ws[jj][cc + 2] +
               p[c0 + cc + 3] * ws[jj][cc + 3];
    }
    if (j0 + jj < Fh) dh[i * Fh + j0 + jj] = acc;
  }
  __syncthreads();
  for (int g = 0; g < ng; ++g) {
    const int r0 = node_off[g0 + g], rows = node_off[g0 + g + 1] - r0;
    float* __restrict__ out = dH + (int64_t)r0 * Fh;
    for (int e = t; e < rows * Fh; e += 256) out[e] = dh[g * Fh + e % Fh];
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

inline int pad4(int x) { return (x + 3) & ~3; }

// dhead_W [Kd, N] = A^T D over `rows` rows, A [rows, Kd] and D with row pitch pad4(N): the tensor-core TN kernel takes
// Kd <= 128 and N % 4 == 0, so the contraction runs 128 result rows at a time into Wpad [Kd, pad4(N)], whose N real
// columns are then copied to dW.  tn_part holds head_weight_grad_partial_floats(rows, Kd, N) floats.
size_t head_weight_grad_partial_floats(int rows, int Kd, int N) {
  GemmTNArgs t;
  t.M = rows; t.Kd = std::min(Kd, 128); t.N = pad4(N); t.S = 1;
  return gemm_tn_auto_partial_floats(t);
}

int head_weight_grad(const float* A, int rows, int Kd, const float* D, int N, float* Wpad, float* tn_part, float* dW,
                     cudaStream_t st) {
  const int Np = pad4(N);
  for (int f0 = 0; f0 < Kd; f0 += 128) {
    GemmTNArgs t;
    t.M = rows; t.Kd = std::min(128, Kd - f0); t.N = Np; t.S = 1;
    t.A0 = A + f0; t.lda0 = Kd;
    t.D = D; t.ldd = Np;
    t.out = Wpad + (size_t)f0 * Np; t.partial = tn_part;
    int rc = gemm_tn_auto(t, st);
    if (rc) return rc;
  }
  const int64_t total = (int64_t)Kd * N;
  copy_pitched_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(Wpad, Np, dW, N, Kd, N);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

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
    GemmTNArgs t;  // ddense_W
    t.M = (int)B; t.Kd = Fh; t.N = Fm; t.S = 1;
    w.tn_part = c.take(std::max(head_weight_grad_partial_floats((int)B, Fm, Nt), gemm_tn_auto_partial_floats(t)));
    w.splitk = c.take((size_t)8 * B * std::max(Fm, Fh));  // split-K partial sums of the two long contractions
  }
  w.bytes = c.bytes;
  return w;
}

// Parameter gradients of agcn_head_loss_grad_ex
struct HeadGrads {
  float *dH, *ddense_W, *ddense_b, *dhead_W, *dhead_b;
};

// Both head calls.  The forward runs the same kernels with the same tile configurations for training (grads set) and
// prediction (grads NULL): gather, dense product and tanh in head_fwd_kernel, the logits on the tensor cores with the
// loss (or the probabilities) in their epilogue, the single-task softmax in softmax_ce_kernel.  The evaluation loss is
// therefore bit-identical to the training loss.  Prediction writes the probabilities (weighted L2: the values) to
// d_probs and the loss to d_loss when targets are given; training writes the loss and every gradient.
//
// Training: the main stream runs dmol = dlog head_W^T and head_bwd_kernel, which ends at dH; the parameter gradients
// run beside it on plan->head.  join_head: `st` waits for them before head_run returns.  Otherwise the caller must make
// `st` wait for plan->ev_head_join before it reads the parameter gradients or ends a capture (agcn_stack_loss_grad).
int head_run(const char* who, const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
             const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights, float scale,
             int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_probs, float* d_loss, const HeadGrads* gr,
             void* d_work, size_t work_bytes, bool join_head, cudaStream_t st) {
  const std::string at = std::string(who) + ": ";
  AGCN_REQUIRE(loss_kind != AGCN_PER_NODE_SOFTMAX_CE,
               at + "AGCN_PER_NODE_SOFTMAX_CE is the per-node head: call agcn_node_head_loss_grad / agcn_node_head_predict");
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
  cudaStream_t side = plan->side, hs = plan->head;

  GemmArgs g_log;
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
  GemmArgs g_dmol;  // split-K partials are left for head_bwd_kernel to add
  g_dmol.M = B; g_dmol.N = Fm; g_dmol.Kd = Nt;
  g_dmol.A0 = w.dlog; g_dmol.lda0 = Ntp;
  g_dmol.B = d_head_W; g_dmol.ldb = Nt; g_dmol.transB = 1;  // head_W is [Fm, Nt] = [N, Kd]
  g_dmol.C = w.dmol; g_dmol.ldc = Fm; g_dmol.split_k_partial = w.splitk; g_dmol.split_k_raw = 1;
  GemmArgs g_dhs;
  g_dhs.M = B; g_dhs.N = Fh; g_dhs.Kd = Fm;
  g_dhs.A0 = w.dmol; g_dhs.lda0 = Fm;
  g_dhs.B = d_dense_W; g_dhs.ldb = Fm; g_dhs.transB = 1;    // dense_W is [Fh, Fm] = [N, Kd]
  g_dhs.C = w.dhsum; g_dhs.ldc = Fh; g_dhs.split_k_partial = w.splitk;
  // dhsum = dpre dense_W^T runs inside head_bwd_kernel, on the CUDA cores, up to 2^26 multiply-adds: every CTA reads all
  // of dense_W, which the large products pay for (B = 4096, Fh = 128, Fm = 512: 637 against 558 us per head call on
  // the tensor cores); those keep the tcgen05 product and a broadcast into dH
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
  // few MFLOP) decides the accuracy of every gradient behind it.  Plain fp32 FMAs keep it at fp32 rounding level;
  // 3xTF32 is ~4x coarser.  w.pre receives tanh'(a).
  {
    const dim3 grid((unsigned)((B + HEAD_GRAPHS - 1) / HEAD_GRAPHS), (unsigned)((Fm + 255) / 256));
    ProfScope prof("head_fwd_kernel", st);
    head_fwd_kernel<<<grid, 256, 0, st>>>(d_H, plan->d_node_off, plan->d_n, d_dense_W, d_dense_b, B, Fh, Fm, w.hsum,
                                          w.pre, w.mol);
  }
  AGCN_LAUNCH_CHECK();
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

  // the head's parameter gradients on plan->head, beside the chain back to dH on the main stream
  AGCN_CUDA(cudaEventRecord(plan->ev_head_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(hs, plan->ev_head_fork, 0));
  weighted_colsum_kernel<<<(Nt + 31) / 32, 256, 0, hs>>>(w.dlog, Ntp, B, Nt, nullptr, gr->dhead_b);
  AGCN_LAUNCH_CHECK();
  if ((rc = head_weight_grad(w.mol, B, Fm, w.dlog, Nt, w.dWh_pad, w.tn_part, gr->dhead_W, hs))) return rc;

  // main stream: dmol = dlog head_W^T, then dpre and dH in head_bwd_kernel (w.dmol := dpre)
  if ((rc = gemm_auto(g_dmol, w.tcC, st, /*presplit=*/true))) return rc;
  {
    const int chunks = tc_dmol ? tc_gemm_ksplit(g_dmol) : 1;
    const size_t smem = (size_t)HEAD_GRAPHS * (Fm + Fh) * sizeof(float);
    if (smem > 32 * 1024)
      AGCN_CUDA(cudaFuncSetAttribute(head_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope prof("head_bwd_kernel", st);
    head_bwd_kernel<<<(unsigned)((B + HEAD_GRAPHS - 1) / HEAD_GRAPHS), 256, smem, st>>>(
        chunks > 1 ? w.splitk : w.dmol, (int64_t)B * Fm, chunks, w.pre, d_dense_W, plan->d_node_off, B, Fh, Fm, w.dmol,
        tc_dhs ? nullptr : gr->dH);
  }
  AGCN_LAUNCH_CHECK();
  if (tc_dhs) {
    if ((rc = tc_gemm(g_dhs, w.tcD, st))) return rc;
    segment_broadcast_kernel<<<(B + 7) / 8, 256, 0, st>>>(w.dhsum, plan->d_node_off, B, Fh, gr->dH);
    AGCN_LAUNCH_CHECK();
  }
  // dense parameter gradients from dpre, behind dhead_W on plan->head (they share tn_part)
  AGCN_CUDA(cudaEventRecord(plan->ev_head_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(hs, plan->ev_head_fork, 0));
  weighted_colsum_kernel<<<(Fm + 31) / 32, 256, 0, hs>>>(w.dmol, Fm, B, Fm, plan->d_n, gr->ddense_b);
  AGCN_LAUNCH_CHECK();
  {
    GemmTNArgs t;  // ddense_W = hsum^T dpre
    t.M = B; t.Kd = Fh; t.N = Fm; t.S = 1;
    t.A0 = w.hsum; t.lda0 = Fh;
    t.D = w.dmol; t.ldd = Fm;
    t.out = gr->ddense_W; t.partial = w.tn_part;
    if ((rc = gemm_tn_auto(t, hs))) return rc;
  }
  AGCN_CUDA(cudaEventRecord(plan->ev_head_join, hs));
  if (join_head) AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_head_join, 0));
  return AGCN_OK;
}

// ---- per-node head (agcn_node_head_*): the logits of every packed row, softmax cross-entropy per row

constexpr int COLSUM_ROWS = 64;  // rows per CTA of colsum_part_kernel

// First stage of dhead_b = colsum(dlog) over the R rows: part[k, c] = sum of M[r, c] over the rows [64 k, 64 k + 64).
// weighted_colsum_kernel would walk all R rows in each of its (C + 31) / 32 CTAs, a serial chain at R = 32 k; here every
// CTA sums 64 rows, threads laid out [row lane][column] as act_bwd_colsum_kernel (coalesced, fixed order), and
// colsum_reduce adds the ceil(R / 64) parts.  Deterministic: no atomics.
__global__ void __launch_bounds__(256) colsum_part_kernel(const float* __restrict__ M, int ld, int64_t R, int C,
                                                          float* __restrict__ part) {
  __shared__ float red[256];
  const int64_t r0 = (int64_t)blockIdx.x * COLSUM_ROWS, r1 = min(R, r0 + COLSUM_ROWS);
  const int cols = min(C, 256), lanes = 256 / cols;
  for (int cbase = 0; cbase < C; cbase += cols) {
    const int c = cbase + (int)(threadIdx.x % cols), rl = threadIdx.x / cols;
    float s = 0.f;
    if (c < C && rl < lanes)
      for (int64_t r = r0 + rl; r < r1; r += lanes) s += M[r * ld + c];
    red[threadIdx.x] = s;
    __syncthreads();
    if (rl == 0 && c < C) {
      for (int l = 1; l < lanes; ++l) s += red[l * cols + (threadIdx.x % cols)];
      part[(int64_t)blockIdx.x * C + c] = s;
    }
    __syncthreads();
  }
}

int colsum_parts(const agcn_plan* plan) { return (int)((plan->R + COLSUM_ROWS - 1) / COLSUM_ROWS); }

// As carve_head: the forward areas are agcn_node_head_predict's whole work area, training adds its areas behind them.
struct NodeHeadWork {
  float *dlog, *loss_part, *tcB;
  float *tcC, *dWh_pad, *tn_part, *colsum_part;
  size_t bytes;
};

NodeHeadWork carve_node_head(const agcn_plan* plan, int Fh, int C, bool train, void* base) {
  Arena c(base);
  const size_t R = (size_t)plan->R;
  const int Cp = pad4(C);
  NodeHeadWork w{};
  w.dlog = c.take(R * Cp);   // row pitch Cp: the logits, overwritten by d loss / d logits in training
  w.loss_part = c.take(R);
  w.tcB = c.take(tc_gemm_scratch_floats(C, Fh, 1, 1));   // head_W      (logits = H head_W)
  if (train) {
    w.tcC = c.take(tc_gemm_scratch_floats(Fh, C, 1, 1));  // head_W^T    (dH = dlog head_W^T)
    w.dWh_pad = c.take((size_t)Fh * Cp);
    w.tn_part = c.take(head_weight_grad_partial_floats((int)R, Fh, C));
    w.colsum_part = c.take((size_t)colsum_parts(plan) * C);
  }
  w.bytes = c.bytes;
  return w;
}

// Both node-head calls: one forward for training (dH set) and prediction, so the evaluation loss is bit-identical to
// the training loss.  Forward: logits GEMM (bias in its epilogue), softmax_ce_kernel over the R rows, loss partials
// summed in fixed order.  Backward: dH = dlog head_W^T on `st`, dhead_W = H^T dlog and dhead_b = colsum(dlog) beside it
// on the side stream.
int node_head_run(const char* who, const agcn_plan* plan, const float* d_H, const float* d_head_W,
                  const float* d_head_b, const float* d_targets, const float* d_weights, float scale, int32_t Fh,
                  int32_t C, float* d_probs, float* d_loss, float* d_dH, float* d_dhead_W, float* d_dhead_b,
                  void* d_work, size_t work_bytes, cudaStream_t st) {
  const std::string at = std::string(who) + ": ";
  AGCN_REQUIRE(Fh >= 1 && C >= 1, at + "unsupported sizes (need Fh >= 1 and C >= 1)");
  const bool train = d_dH != nullptr;
  int rc = plan_use(plan, st);
  if (rc) return rc;
  NodeHeadWork w = carve_node_head(plan, Fh, C, train, d_work);
  if (w.bytes > work_bytes) {
    set_error(at + "workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  const int R = (int)plan->R, Cp = pad4(C);
  cudaStream_t side = plan->side;

  GemmArgs g_log, g_dH;
  g_log.M = R; g_log.N = C; g_log.Kd = Fh;
  g_log.A0 = d_H; g_log.lda0 = Fh;
  g_log.B = d_head_W; g_log.ldb = C;
  g_log.C = w.dlog; g_log.ldc = Cp;
  g_log.bias = d_head_b;
  // dH: contraction over the C classes, R / 128 row tiles -- enough tiles without split-K
  g_dH.M = R; g_dH.N = Fh; g_dH.Kd = C;
  g_dH.A0 = w.dlog; g_dH.lda0 = Cp;
  g_dH.B = d_head_W; g_dH.ldb = C; g_dH.transB = 1;   // head_W is [Fh, C] = [N, Kd]
  g_dH.C = d_dH; g_dH.ldc = Fh;
  const bool tc_log = tc_gemm_supported(g_log), tc_dH = train && tc_gemm_supported(g_dH);

  // parameter operands (hi / lo split, K-major) on the side stream
  AGCN_CUDA(cudaEventRecord(plan->ev_side_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(side, plan->ev_side_fork, 0));
  if (tc_log && (rc = tc_gemm_split_b(g_log, w.tcB, side))) return rc;
  if (tc_dH && (rc = tc_gemm_split_b(g_dH, w.tcC, side))) return rc;
  AGCN_CUDA(cudaEventRecord(plan->ev_side_join, side));
  AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));

  // logits (only the C real columns of dlog are written and read back: the pad columns feed nothing but the pad
  // columns of dWh_pad, which are not copied out), then the row softmax: d loss / d logits in place (training) or the
  // probabilities, and the per-row loss terms
  if ((rc = gemm_auto(g_log, w.tcB, st, /*presplit=*/true))) return rc;
  (train ? softmax_ce_kernel<true> : softmax_ce_kernel<false>)<<<(R + 7) / 8, 256, 0, st>>>(
      w.dlog, Cp, d_targets, d_weights, R, C, scale, d_probs, w.loss_part);
  AGCN_LAUNCH_CHECK();
  if (d_loss) {
    sum_parts_kernel<<<1, 256, 0, st>>>(w.loss_part, R, d_loss);
    AGCN_LAUNCH_CHECK();
  }
  if (!train) return AGCN_OK;

  // parameter gradients on the side stream, beside dH on the main stream
  AGCN_CUDA(cudaEventRecord(plan->ev_side_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(side, plan->ev_side_fork, 0));
  colsum_part_kernel<<<colsum_parts(plan), 256, 0, side>>>(w.dlog, Cp, R, C, w.colsum_part);
  AGCN_LAUNCH_CHECK();
  if ((rc = colsum_reduce(w.colsum_part, colsum_parts(plan), C, d_dhead_b, side))) return rc;
  if ((rc = head_weight_grad(d_H, R, Fh, w.dlog, C, w.dWh_pad, w.tn_part, d_dhead_W, side))) return rc;
  AGCN_CUDA(cudaEventRecord(plan->ev_side_join, side));

  if ((rc = gemm_auto(g_dH, w.tcC, st, /*presplit=*/true))) return rc;
  AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));
  return AGCN_OK;
}

}  // namespace

int head_loss_grad(const agcn_plan* plan, const float* d_H, const float* d_dense_W, const float* d_dense_b,
                   const float* d_head_W, const float* d_head_b, const float* d_targets, const float* d_weights,
                   float scale, int32_t loss_kind, int32_t Fh, int32_t Fm, int32_t Nt, float* d_loss, float* d_dH,
                   float* d_ddense_W, float* d_ddense_b, float* d_dhead_W, float* d_dhead_b, void* d_work,
                   size_t work_bytes, bool join_head, cudaStream_t st) {
  AGCN_REQUIRE(plan && d_H && d_dense_W && d_dense_b && d_head_W && d_head_b && d_targets && d_weights && d_loss &&
                   d_dH && d_ddense_W && d_ddense_b && d_dhead_W && d_dhead_b && d_work,
               "head_loss_grad: null pointer");
  const HeadGrads gr{d_dH, d_ddense_W, d_ddense_b, d_dhead_W, d_dhead_b};
  return head_run("head_loss_grad", plan, d_H, d_dense_W, d_dense_b, d_head_W, d_head_b, d_targets, d_weights, scale,
                  loss_kind, Fh, Fm, Nt, nullptr, d_loss, &gr, d_work, work_bytes, join_head, st);
}

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
  return head_loss_grad(plan, d_H, d_dense_W, d_dense_b, d_head_W, d_head_b, d_targets, d_weights, scale, loss_kind, Fh,
                        Fm, Nt, d_loss, d_dH, d_ddense_W, d_ddense_b, d_dhead_W, d_dhead_b, d_work, work_bytes,
                        /*join_head=*/true, (cudaStream_t)stream);
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
                  loss_kind, Fh, Fm, Nt, d_probs, d_loss, nullptr, d_work, work_bytes, true, (cudaStream_t)stream);
}

int agcn_node_head_workspace_bytes(const agcn_plan* plan, int32_t Fh, int32_t C, size_t* bytes) {
  AGCN_REQUIRE(plan && bytes && Fh >= 1 && C >= 1, "node_head_workspace_bytes: bad arguments");
  *bytes = carve_node_head(plan, Fh, C, true, nullptr).bytes + 256;
  return AGCN_OK;
}

int agcn_node_head_loss_grad(const agcn_plan* plan, const float* d_H, const float* d_head_W, const float* d_head_b,
                             const float* d_targets, const float* d_weights, float scale, int32_t Fh, int32_t C,
                             float* d_loss, float* d_dH, float* d_dhead_W, float* d_dhead_b, void* d_work,
                             size_t work_bytes, void* stream) {
  AGCN_REQUIRE(plan && d_H && d_head_W && d_head_b && d_targets && d_weights && d_loss && d_dH && d_dhead_W &&
                   d_dhead_b && d_work,
               "node_head_loss_grad: null pointer");
  return node_head_run("node_head_loss_grad", plan, d_H, d_head_W, d_head_b, d_targets, d_weights, scale, Fh, C,
                       nullptr, d_loss, d_dH, d_dhead_W, d_dhead_b, d_work, work_bytes, (cudaStream_t)stream);
}

int agcn_node_head_predict_workspace_bytes(const agcn_plan* plan, int32_t Fh, int32_t C, size_t* bytes) {
  AGCN_REQUIRE(plan && bytes && Fh >= 1 && C >= 1, "node_head_predict_workspace_bytes: bad arguments");
  *bytes = carve_node_head(plan, Fh, C, false, nullptr).bytes + 256;
  return AGCN_OK;
}

int agcn_node_head_predict(const agcn_plan* plan, const float* d_H, const float* d_head_W, const float* d_head_b,
                           const float* d_targets, const float* d_weights, float scale, int32_t Fh, int32_t C,
                           float* d_probs, float* d_loss, void* d_work, size_t work_bytes, void* stream) {
  AGCN_REQUIRE(!d_targets == !d_weights && !d_targets == !d_loss,
               "node_head_predict: d_targets, d_weights and d_loss must be all NULL or all set");
  AGCN_REQUIRE(plan && d_H && d_head_W && d_head_b && d_probs && d_work, "node_head_predict: null pointer");
  return node_head_run("node_head_predict", plan, d_H, d_head_W, d_head_b, d_targets, d_weights, scale, Fh, C, d_probs,
                       d_loss, nullptr, nullptr, nullptr, d_work, work_bytes, (cudaStream_t)stream);
}

}  // extern "C"
