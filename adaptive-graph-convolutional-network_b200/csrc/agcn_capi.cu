// C ABI of the SGC-LL layer (include/agcn_sgcll.h): orchestration of the node-level GEMMs and the
// per-graph kernels for one whole batch.  Reference: models/layers/graphconv.py:85-252,
// models/layers/graphconv_reslap.py:45-230.
#include <algorithm>

#include "agcn_internal.cuh"

using namespace agcn;

namespace {

// node-level GEMM: tensor cores when the operands are TMA-compatible, CUDA cores otherwise (F = 75)
int node_gemm_tn(const GemmTNArgs& t, cudaStream_t st) {
  if (tc_gemm_tn_supported(t)) return tc_gemm_tn(t, st);
  return gemm_tn(t, st);
}

// presplit: the hi / lo copies of B in tc_scratch were already produced by tc_gemm_split_b (side stream)
int node_gemm(const GemmArgs& g, float* tc_scratch, cudaStream_t st, bool presplit = false) {
  if (tc_gemm_supported(g)) {
    if (!presplit) {
      int rc = tc_gemm_split_b(g, tc_scratch, st);
      if (rc) return rc;
    }
    return tc_gemm(g, tc_scratch, st);
  }
  return gemm_rows(g, st);
}

// Y = act(sum_k T_k W_k + b)   graphconv.py:238-247, :118-123
GemmArgs y_gemm_args(const agcn_sgcll_desc* d, int R, const float* X, const float* T, const float* weight,
                     const float* bias, float* Y) {
  GemmArgs g;
  g.M = R; g.N = d->Fo; g.Kd = d->F; g.S = d->K;
  g.A0 = X; g.lda0 = d->F;
  g.A1 = T; g.lda1 = d->F; g.sliceA1 = (int64_t)R * d->F;
  g.B = weight; g.ldb = d->K * d->Fo; g.sliceB = d->Fo;
  g.C = Y; g.ldc = d->Fo;
  g.bias = bias; g.act = d->activation;
  return g;
}

// G_k = dYpre W_k^T   (K == 1: this is dX)
GemmArgs g_gemm_args(const agcn_sgcll_desc* d, int R, const float* dYp, const float* weight, float* C) {
  GemmArgs g;
  g.M = R; g.N = d->F; g.Kd = d->Fo; g.Z = d->K;
  g.A0 = dYp; g.lda0 = d->Fo;
  g.B = weight; g.ldb = d->K * d->Fo; g.sliceB = d->Fo; g.transB = 1;
  g.C = C; g.ldc = d->F; g.sliceC = (int64_t)R * d->F;
  return g;
}

struct Modes {
  bool shortcut, paper, reslap, full, need_dL;
};

Modes modes_of(const agcn_sgcll_desc* d) {
  Modes m;
  m.shortcut = literal_shortcut(d->variant, d->laplacian_mode);
  m.paper = d->laplacian_mode == AGCN_LAP_PAPER;
  m.reslap = d->variant == AGCN_VARIANT_SGC_LL_RESLAP;
  m.full = m.paper && d->metric_grad == AGCN_METRIC_GRAD_FULL;
  m.need_dL = !m.shortcut;
  return m;
}

// saved area layout (forward -> backward)
struct Saved {
  float *T, *Lall, *dist, *dis, *stats, *XW, *tcG, *ftG;
  size_t bytes;
};

Saved carve_saved(const agcn_sgcll_desc* d, const agcn_plan* p, void* base) {
  const Modes m = modes_of(d);
  Arena c(base);
  Saved s{};
  s.T = c.take((size_t)(d->K > 1 ? d->K - 1 : 0) * p->R * d->F);
  s.Lall = m.shortcut ? nullptr : c.take((size_t)p->LL);
  s.dist = m.paper ? c.take((size_t)p->LL) : nullptr;
  s.dis = m.paper ? c.take((size_t)p->R) : nullptr;
  s.stats = m.shortcut ? nullptr : c.take((size_t)4 * p->B);
  s.XW = m.full ? c.take((size_t)p->R * d->F) : nullptr;
  s.tcG = c.take(tc_gemm_scratch_floats(d->F, d->Fo, 1, d->K));  // hi / lo of W_k^T for the backward G GEMM
  s.ftG = c.take(fused_w_floats(d->F, d->Fo, d->K));             // the same operand in the fused backward's layout
  s.bytes = c.bytes;
  return s;
}

// dL_all of the per-graph recurrences is accumulated by several CTAs per graph (one per group of feature chunks), each
// writing its own partial matrix: up to 8 parts as long as the scratch stays below 1 GB
inline int64_t dl_stride(const agcn_plan* p) { return (p->LL + 63) & ~(int64_t)63; }
inline int dl_parts(const agcn_sgcll_desc* d, const agcn_plan* p) {
  if (d->K < 2) return 1;
  int parts = std::min(8, (d->F + 31) / 32);
  while (parts > 1 && (int64_t)parts * dl_stride(p) * 4 > ((int64_t)1 << 30)) --parts;
  return std::max(1, parts);
}

struct Work {
  float *XW, *dYp, *G, *V, *tn_part, *act_part, *dL, *dXW, *dalpha_part, *dbeta_part, *tcY, *tcM, *big, *ftY;
  size_t bytes;
};

Work carve_work(const agcn_sgcll_desc* d, const agcn_plan* p, void* base) {
  const Modes m = modes_of(d);
  Arena c(base);
  Work w{};
  w.XW = c.take((size_t)p->R * d->F);  // forward: X M_L (when the similarity is needed and not saved)
  w.dYp = c.take((size_t)p->R * d->Fo);
  w.G = c.take((size_t)d->K * p->R * d->F);
  w.V = c.take((size_t)(d->K > 1 ? d->K - 1 : 0) * p->R * d->Fo);  // V_k = T_k(L^T) dYpre of the recurrence-first backward
  size_t tn = gemm_tn_partial_floats((int)p->R, d->F, d->Fo, d->K);
  if (m.full) tn = std::max(tn, gemm_tn_partial_floats((int)p->R, d->F, d->F, 1));
  {
    GemmTNArgs t;
    t.M = (int)p->R; t.Kd = d->F; t.N = d->Fo; t.S = d->K;
    tn = std::max(tn, tc_gemm_tn_partial_floats(t));
    t.N = d->F; t.S = 1;
    tn = std::max(tn, tc_gemm_tn_partial_floats(t));
  }
  w.tn_part = c.take(tn);
  w.act_part = c.take(act_bwd_partial_floats(p->R, d->Fo));
  w.dL = m.need_dL ? c.take((size_t)dl_parts(d, p) * dl_stride(p)) : nullptr;
  w.dXW = m.full ? c.take((size_t)p->R * d->F) : nullptr;
  w.dalpha_part = c.take((size_t)p->B);
  w.dbeta_part = c.take((size_t)p->B);
  // hi / lo copies of the parameter operands of the tensor-core GEMMs
  w.tcY = c.take(tc_gemm_scratch_floats(d->Fo, d->F, d->K, 1));
  w.tcM = c.take(tc_gemm_scratch_floats(d->F, d->F, 1, 1));
  w.big = c.take(big_work_floats(p, m.full));  // sweeps of the graphs with n > AGCN_SMALL_MAX
  w.ftY = c.take(fused_w_floats(d->Fo, d->F, d->K));  // pre-split W_k of the fused forward kernel
  w.bytes = c.bytes;
  return w;
}

int check_desc(const agcn_sgcll_desc* d, const agcn_plan* p) {
  AGCN_REQUIRE(d && p, "null desc or plan");
  AGCN_REQUIRE(d->F >= 1 && d->Fo >= 1 && d->K >= 1, "F, Fo, K must be >= 1");
  AGCN_REQUIRE(d->variant == AGCN_VARIANT_SGC_LL || d->variant == AGCN_VARIANT_SGC_LL_RESLAP, "unknown variant");
  AGCN_REQUIRE(d->laplacian_mode == AGCN_LAP_REFERENCE_LITERAL || d->laplacian_mode == AGCN_LAP_PAPER,
               "unknown laplacian_mode");
  AGCN_REQUIRE(d->metric_grad == AGCN_METRIC_GRAD_REFERENCE || d->metric_grad == AGCN_METRIC_GRAD_FULL,
               "unknown metric_grad");
  AGCN_REQUIRE(d->activation == AGCN_ACT_LINEAR || d->activation == AGCN_ACT_RELU, "unknown activation");
  AGCN_REQUIRE(p->R < (1ll << 31) / std::max(d->F, d->Fo), "batch too large for 32-bit row indexing");
  return AGCN_OK;
}

}  // namespace

namespace {

// ------------------------------------------------------------------------------------------------
// Feature padding.  75 atom features (the first layer of every molecule network) are neither a multiple of 4 (no
// 16-byte row accesses) nor of 32 (no TMA row tiles): the layer then ran on the scalar / generic kernels and cost twice
// a hidden layer (profiles/r02p_timeline_c2.txt: 60 + 38 us against 22 + 24 us).  With the literal shortcut (no metric
// block, M_L unused) the layer is LINEAR in the feature columns, so it runs on zero-padded copies instead: X -> [R, Fp],
// weight -> [Fp K, Fo] (rows f K + k of the padded features are zero), Fp = F rounded up to 32.  T_k, dweight and dX of
// the padded problem contain the unpadded ones as their leading columns / rows.
// ------------------------------------------------------------------------------------------------
int padded_features(const agcn_sgcll_desc* d, const agcn_plan* p) {
  const int F = d->F;
  if (F < 33 || F % 32 == 0) return F;
  if (!literal_shortcut(d->variant, d->laplacian_mode)) return F;
  if (d->flags & (AGCN_OUT_RES_L | AGCN_OUT_RES_W | AGCN_OUT_L_ALL)) return F;
  const int Fp = (F + 31) & ~31;
  if (!fused_fwd_supported(p, Fp, d->Fo, d->K)) return F;
  return Fp;
}

struct PadSaved {
  float *Xp, *Wp;
  void* inner;
  size_t bytes;
};
PadSaved carve_pad_saved(const agcn_sgcll_desc* d2, const agcn_plan* p, void* base) {
  Arena c(base);
  PadSaved s{};
  s.Xp = c.take((size_t)p->R * d2->F);
  s.Wp = c.take((size_t)d2->F * d2->K * d2->Fo);
  s.inner = c.area(carve_saved(d2, p, nullptr).bytes + 256);
  s.bytes = c.bytes;
  return s;
}
struct PadWork {
  float *dXp, *dWp, *dMp;
  void* inner;
  size_t inner_bytes, bytes;
};
PadWork carve_pad_work(const agcn_sgcll_desc* d2, const agcn_plan* p, void* base) {
  Arena c(base);
  PadWork w{};
  w.dXp = c.take((size_t)p->R * d2->F);
  w.dWp = c.take((size_t)d2->F * d2->K * d2->Fo);
  w.dMp = c.take((size_t)d2->F * d2->F);
  w.inner_bytes = carve_work(d2, p, nullptr).bytes + 256;
  w.inner = c.area(w.inner_bytes);
  w.bytes = c.bytes;
  return w;
}

// agcn_sgcll_forward_host's scratch: the padded wire layouts of X, L and Y, their packed copies, the layer's areas
struct HostScratch {
  float *Xpad, *Lpad, *Ypad, *X, *L, *Y;
  void *saved, *work;
  size_t work_bytes, bytes;
};
HostScratch carve_host(const agcn_sgcll_desc* d, const agcn_plan* p, void* base) {
  size_t saved = 0;
  Arena c(base);
  HostScratch h{};
  agcn_sgcll_workspace_bytes(d, p, &saved, &h.work_bytes);
  const size_t B = p->B, N = p->Nmax;
  h.Xpad = c.take(B * N * d->F);
  h.Lpad = c.take(B * N * N);
  h.Ypad = c.take(B * N * d->Fo);
  h.X = c.take((size_t)p->R * d->F);
  h.L = c.take((size_t)p->LL);
  h.Y = c.take((size_t)p->R * d->Fo);
  h.saved = c.area(saved);
  h.work = c.area(h.work_bytes);
  h.bytes = c.bytes;
  return h;
}

// dst[r, c] = c < Fs ? src[r, c] : 0   (rows x Fd)
__global__ void pad_cols_kernel(const float* __restrict__ src, int Fs, float* __restrict__ dst, int Fd, long long rows) {
  const long long total = rows * Fd;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / Fd;
    const int c = (int)(e - r * Fd);
    dst[e] = c < Fs ? src[r * Fs + c] : 0.f;
  }
}
// dst[r, c] = src[r, c] for c < Fd   (rows x Fd out of rows x Fs)
__global__ void unpad_cols_kernel(const float* __restrict__ src, int Fs, float* __restrict__ dst, int Fd, long long rows) {
  const long long total = rows * Fd;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / Fd;
    const int c = (int)(e - r * Fd);
    dst[e] = src[r * Fs + c];
  }
}
// dst[0 .. n_copy) = src, dst[n_copy .. n_total) = 0
__global__ void copy_then_zero_kernel(const float* __restrict__ src, float* __restrict__ dst, long long n_copy, long long n_total) {
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_total; e += (long long)gridDim.x * blockDim.x)
    dst[e] = e < n_copy ? src[e] : 0.f;
}
inline unsigned grid_for(long long total) { return (unsigned)std::max<long long>(1, std::min<long long>((total + 255) / 256, 1184)); }

int forward_impl(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                 const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_bias,
                 const float* d_alpha, const float* d_beta, float* d_Y, float* d_resL, float* d_resW, float* d_Lall,
                 void* d_saved, void* d_work, size_t work_bytes, void* stream);
int backward_impl(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                  const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_alpha,
                  const float* d_beta, const float* d_Y, const float* d_dY, const float* d_dLall_in, const void* d_saved,
                  float* d_dX, float* d_dM_L, float* d_dweight, float* d_dbias, float* d_dalpha, float* d_dbeta,
                  float* d_dLprev, void* d_work, size_t work_bytes, void* stream);

}  // namespace

extern "C" {

int agcn_sgcll_workspace_bytes(const agcn_sgcll_desc* desc, const agcn_plan* plan, size_t* saved_bytes,
                               size_t* work_bytes) {
  AGCN_REQUIRE(desc && plan, "null desc or plan");
  const int Fp = padded_features(desc, plan);
  if (Fp != desc->F) {
    agcn_sgcll_desc d2 = *desc;
    d2.F = Fp;
    if (saved_bytes) *saved_bytes = carve_pad_saved(&d2, plan, nullptr).bytes + 256;
    if (work_bytes) *work_bytes = carve_pad_work(&d2, plan, nullptr).bytes + 256;
    return AGCN_OK;
  }
  if (saved_bytes) *saved_bytes = carve_saved(desc, plan, nullptr).bytes + 256;
  if (work_bytes) *work_bytes = carve_work(desc, plan, nullptr).bytes + 256;
  return AGCN_OK;
}

int agcn_sgcll_forward(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                       const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_bias,
                       const float* d_alpha, const float* d_beta, float* d_Y, float* d_resL, float* d_resW,
                       float* d_Lall, void* d_saved, void* d_work, size_t work_bytes, void* stream) {
  int rc = check_desc(desc, plan);
  if (rc) return rc;
  const int Fp = padded_features(desc, plan);
  if (Fp == desc->F)
    return forward_impl(desc, plan, d_X, d_Lint, d_Lprev, d_M_L, d_weight, d_bias, d_alpha, d_beta, d_Y, d_resL, d_resW,
                        d_Lall, d_saved, d_work, work_bytes, stream);
  AGCN_REQUIRE(d_X && d_weight && d_saved && d_work, "forward: null pointer");
  agcn_sgcll_desc d2 = *desc;
  d2.F = Fp;
  PadSaved ps = carve_pad_saved(&d2, plan, d_saved);
  PadWork pw = carve_pad_work(&d2, plan, d_work);
  if (pw.bytes > work_bytes) {
    set_error("forward: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = plan_use(plan, st))) return rc;
  pad_cols_kernel<<<grid_for((long long)plan->R * Fp), 256, 0, st>>>(d_X, desc->F, ps.Xp, Fp, plan->R);
  AGCN_LAUNCH_CHECK();
  {
    const long long n_copy = (long long)desc->F * desc->K * desc->Fo, n_total = (long long)Fp * desc->K * desc->Fo;
    copy_then_zero_kernel<<<grid_for(n_total), 256, 0, st>>>(d_weight, ps.Wp, n_copy, n_total);
    AGCN_LAUNCH_CHECK();
  }
  // M_L is not read in the literal shortcut (no similarity matrix is built): the impl only checks the pointer
  return forward_impl(&d2, plan, ps.Xp, d_Lint, d_Lprev, d_M_L, ps.Wp, d_bias, d_alpha, d_beta, d_Y, d_resL, d_resW, d_Lall,
                      ps.inner, pw.inner, pw.inner_bytes, stream);
}

int agcn_sgcll_backward(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                        const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_alpha,
                        const float* d_beta, const float* d_Y, const float* d_dY, const float* d_dLall_in,
                        const void* d_saved, float* d_dX, float* d_dM_L, float* d_dweight, float* d_dbias,
                        float* d_dalpha, float* d_dbeta, float* d_dLprev, void* d_work, size_t work_bytes,
                        void* stream) {
  int rc = check_desc(desc, plan);
  if (rc) return rc;
  const int Fp = padded_features(desc, plan);
  if (Fp == desc->F)
    return backward_impl(desc, plan, d_X, d_Lint, d_Lprev, d_M_L, d_weight, d_alpha, d_beta, d_Y, d_dY, d_dLall_in, d_saved,
                         d_dX, d_dM_L, d_dweight, d_dbias, d_dalpha, d_dbeta, d_dLprev, d_work, work_bytes, stream);
  AGCN_REQUIRE(d_saved && d_work && d_dM_L && d_dweight, "backward: null pointer");
  agcn_sgcll_desc d2 = *desc;
  d2.F = Fp;
  PadSaved ps = carve_pad_saved(&d2, plan, const_cast<void*>(d_saved));
  PadWork pw = carve_pad_work(&d2, plan, d_work);
  if (pw.bytes > work_bytes) {
    set_error("backward: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // the padded problem on the copies the forward pass saved; its gradients hold the real ones as leading rows / columns
  rc = backward_impl(&d2, plan, ps.Xp, d_Lint, d_Lprev, d_M_L, ps.Wp, d_alpha, d_beta, d_Y, d_dY, d_dLall_in, ps.inner,
                     d_dX ? pw.dXp : nullptr, pw.dMp, pw.dWp, d_dbias, d_dalpha, d_dbeta, d_dLprev, pw.inner, pw.inner_bytes,
                     stream);
  if (rc) return rc;
  {
    const long long n = (long long)desc->F * desc->K * desc->Fo;   // rows f K + k with f < F: a prefix of the padded dweight
    copy_then_zero_kernel<<<grid_for(n), 256, 0, st>>>(pw.dWp, d_dweight, n, n);
    AGCN_LAUNCH_CHECK();
  }
  if ((rc = zero_async(d_dM_L, (size_t)desc->F * desc->F, st))) return rc;   // tf.py_func has no gradient
  if (d_dX) {
    unpad_cols_kernel<<<grid_for((long long)plan->R * desc->F), 256, 0, st>>>(pw.dXp, Fp, d_dX, desc->F, plan->R);
    AGCN_LAUNCH_CHECK();
  }
  return AGCN_OK;
}

}  // extern "C"

namespace {

int forward_impl(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                       const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_bias,
                       const float* d_alpha, const float* d_beta, float* d_Y, float* d_resL, float* d_resW,
                       float* d_Lall, void* d_saved, void* d_work, size_t work_bytes, void* stream) {
  int rc = check_desc(desc, plan);
  if (rc) return rc;
  AGCN_REQUIRE(d_X && d_Lint && d_M_L && d_weight && d_bias && d_alpha && d_Y && d_saved && d_work,
               "forward: null pointer");
  const Modes m = modes_of(desc);
  AGCN_REQUIRE(!m.reslap || d_beta, "forward: beta required for SGC_LL_Reslap");
  AGCN_REQUIRE(!(desc->flags & AGCN_OUT_RES_L) || d_resL, "forward: d_resL missing");
  AGCN_REQUIRE(!(desc->flags & AGCN_OUT_RES_W) || d_resW, "forward: d_resW missing");
  AGCN_REQUIRE(!(desc->flags & AGCN_OUT_L_ALL) || d_Lall, "forward: d_Lall missing");
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = plan_use(plan, st))) return rc;
  Saved sv = carve_saved(desc, plan, d_saved);
  Work wk = carve_work(desc, plan, d_work);
  if (wk.bytes > work_bytes) {
    set_error("forward: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  const int F = desc->F, Fo = desc->Fo, K = desc->K;
  const int R = (int)plan->R;
  const bool want_resL = desc->flags & AGCN_OUT_RES_L, want_resW = desc->flags & AGCN_OUT_RES_W;
  const bool want_Lall = desc->flags & AGCN_OUT_L_ALL;
  const bool need_W = m.paper || want_resW;
  const bool need_build = !m.shortcut || want_resL || want_resW || want_Lall;
  float* XW = m.full ? sv.XW : wk.XW;

  // the parameter operands of the two big node-level GEMMs (this forward's Y and the backward's G) are
  // rearranged / split on the side stream while the per-graph kernels run
  // Tile path: CUDA-core recurrences (agcn_cheb_tile.cu) + one tensor-core contraction over all rows (agcn_pre_tile.cu)
  const bool fuse_f = fused_fwd_supported(plan, F, Fo, K);
  const bool fuse_b = (desc->flags & AGCN_SAVE_FOR_BACKWARD) && !m.need_dL && fused_bwd_supported(plan, F, Fo, K);
  GemmArgs gy = y_gemm_args(desc, R, d_X, sv.T, d_weight, d_bias, d_Y);
  const bool y_tc = !fuse_f && tc_gemm_supported(gy);
  GemmArgs gg = g_gemm_args(desc, R, d_Y /* placeholder with the alignment of dYpre */, d_weight, wk.G);
  const bool g_tc = !fuse_b && (desc->flags & AGCN_SAVE_FOR_BACKWARD) && tc_gemm_supported(gg);
  if (y_tc || g_tc || fuse_f || fuse_b) {
    AGCN_CUDA(cudaEventRecord(plan->ev_side_fork, st));
    AGCN_CUDA(cudaStreamWaitEvent(plan->side, plan->ev_side_fork, 0));
    if (fuse_f && (rc = fused_fwd_prep(d_weight, F, Fo, K, wk.ftY, plan->side))) return rc;
    if (y_tc && (rc = tc_gemm_split_b(gy, wk.tcY, plan->side))) return rc;
    if (fuse_b && (rc = fused_bwd_prep(d_weight, F, Fo, K, sv.ftG, plan->side))) return rc;
    if (g_tc && (rc = tc_gemm_split_b(gg, sv.tcG, plan->side))) return rc;
    AGCN_CUDA(cudaEventRecord(plan->ev_side_join, plan->side));
  }
  if (need_W) {  // x_w = np.dot(x, M)   graphconv.py:164
    GemmArgs g;
    g.M = R; g.N = F; g.Kd = F;
    g.A0 = d_X; g.lda0 = F;
    g.B = d_M_L; g.ldb = F;
    g.C = XW; g.ldc = F;
    if ((rc = node_gemm(g, wk.tcM, st))) return rc;
  }
  GraphArgs ga;
  ga.plan = plan; ga.F = F; ga.K = K;
  ga.variant = desc->variant; ga.lap_mode = desc->laplacian_mode; ga.metric_full = m.full;
  ga.X = d_X; ga.XW = XW; ga.Lint = d_Lint; ga.Lprev = m.reslap ? d_Lprev : nullptr;
  ga.alpha = d_alpha; ga.beta = d_beta;
  ga.T = sv.T;
  if (need_build) {
    ga.Lall = m.shortcut ? nullptr : sv.Lall;
    ga.Lall_out = want_Lall ? d_Lall : nullptr;
    ga.resL = want_resL ? d_resL : nullptr;
    ga.resW = want_resW ? d_resW : nullptr;
    ga.dist = sv.dist; ga.dis = sv.dis; ga.stats = sv.stats;
    ga.big_work = wk.big;
    if ((rc = graph_build_laplacian(ga, need_W, st))) return rc;
  }
  ga.Lall = m.shortcut ? nullptr : sv.Lall;
  if (fuse_f) {
    // Recurrences on the CUDA cores (agcn_cheb_tile.cu: small-graph tiles on this stream, mid-size graphs and the
    // row-tiled products of the graphs above cheb_small_max on plan->big), then ONE tensor-core contraction over every
    // packed row (agcn_pre_tile.cu): Y = act(sum_k T_k W_k + b)
    const float* Lf = m.shortcut ? d_Lint : sv.Lall;
    const int ident = m.shortcut ? 1 : 0;
    const bool other = cheb_tiles_has_mid(plan) || plan->large_tiles > 0;
    if (other) {
      AGCN_CUDA(cudaEventRecord(plan->ev_big_fork, st));
      AGCN_CUDA(cudaStreamWaitEvent(plan->big, plan->ev_big_fork, 0));
    }
    if ((rc = cheb_tiles_forward(plan, d_X, Lf, ident, F, K, sv.T, st, plan->big))) return rc;
    if (plan->large_tiles > 0 && (rc = graph_chebyshev_fwd(ga, plan->big, AGCN_SMALL_MAX))) return rc;
    if (other) {
      AGCN_CUDA(cudaEventRecord(plan->ev_big_join, plan->big));
      AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_big_join, 0));
    }
    AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));
    return pre_forward(plan, -1, 0, d_X, sv.T, wk.ftY, d_bias, desc->activation, F, Fo, K, d_Y, st);
  }
  if ((rc = graph_chebyshev_fwd(ga, st))) return rc;  // graphconv.py:221-236
  if (y_tc || g_tc || fuse_b) AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));
  // x = reshape(transpose(stack T)) . weight + bias, activation   graphconv.py:238-247, :118-123
  if ((rc = node_gemm(gy, wk.tcY, st, /*presplit=*/true))) return rc;
  return AGCN_OK;
}

int backward_impl(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* d_X, const float* d_Lint,
                  const float* d_Lprev, const float* d_M_L, const float* d_weight, const float* d_alpha,
                  const float* d_beta, const float* d_Y, const float* d_dY, const float* d_dLall_in, const void* d_saved,
                  float* d_dX, float* d_dM_L, float* d_dweight, float* d_dbias, float* d_dalpha, float* d_dbeta,
                  float* d_dLprev, void* d_work, size_t work_bytes, void* stream) {
  int rc = check_desc(desc, plan);
  if (rc) return rc;
  AGCN_REQUIRE(d_X && d_Lint && d_M_L && d_weight && d_alpha && d_Y && d_dY && d_saved && d_work,
               "backward: null input pointer");
  AGCN_REQUIRE(d_dM_L && d_dweight && d_dbias && d_dalpha, "backward: null output pointer");
  const Modes m = modes_of(desc);
  AGCN_REQUIRE(!m.reslap || (d_beta && d_dbeta), "backward: beta / dbeta required for SGC_LL_Reslap");
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = plan_use(plan, st))) return rc;
  Saved sv = carve_saved(desc, plan, const_cast<void*>(d_saved));
  Work wk = carve_work(desc, plan, d_work);
  if (wk.bytes > work_bytes) {
    set_error("backward: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  const int F = desc->F, Fo = desc->Fo, K = desc->K;
  const int R = (int)plan->R;
  const bool has_prev = m.reslap && d_Lprev;

  // d_dX == NULL: the caller does not need the gradient w.r.t. the node features (first layer)
  const bool fuse_b = (desc->flags & AGCN_SAVE_FOR_BACKWARD) && !m.need_dL && d_dX != nullptr &&
                      fused_bwd_supported(plan, F, Fo, K);
  // Recurrence-first dX chain (batches whose graphs all take the recurrence tiles): V_k = T_k(L^T) dYpre on the CUDA cores,
  // then dX = sum_k V_k W_k^T as ONE accumulator on the tensor cores -- the mirror image of the forward pass, same
  // kernels (T_k(L)^T = T_k(L^T)).  Against G_z = dYpre W_z^T followed by the reverse recurrence it needs one TMEM
  // accumulator instead of K (two contraction CTAs per SM: one wave for a batch of 155 row tiles) and reads / writes
  // (K-1) [R, Fo] matrices instead of K [R, F] ones.  Row-tiled graphs (point clouds) keep the G_z form: their products
  // are the expensive part and G_z keeps them F wide.
  const bool vfirst = fuse_b && plan->large_tiles == 0;
  const bool need_G = !fuse_b && (d_dX != nullptr || (m.need_dL && K >= 2));
  // dYpre = dY * act'(Y) and per-CTA column sums; dbias = colsum(dYpre).  The parameter gradients depend on
  // dYpre only -> side stream, overlapping the dX chain.  The fused dX kernel applies act' itself, so in that case
  // (and when the main stream has no use for dYpre at all) the whole dYpre branch lives on the side stream.
  const float* dYp = (desc->activation == AGCN_ACT_RELU) ? wk.dYp : d_dY;
  const bool act_on_side = !vfirst && (fuse_b || (!need_G && !m.need_dL));   // vfirst: the main chain starts from dYpre
  if (!act_on_side && (rc = act_bwd_partials(d_dY, d_Y, wk.dYp, wk.act_part, R, Fo, desc->activation, st))) return rc;
  AGCN_CUDA(cudaEventRecord(plan->ev_side_fork, st));
  AGCN_CUDA(cudaStreamWaitEvent(plan->side, plan->ev_side_fork, 0));
  if (act_on_side && (rc = act_bwd_partials(d_dY, d_Y, wk.dYp, wk.act_part, R, Fo, desc->activation, plan->side)))
    return rc;
  if ((rc = act_bwd_reduce(wk.act_part, d_dbias, R, Fo, plan->side))) return rc;
  float* dXbuf = d_dX ? d_dX : wk.G;  // scratch target when dX itself is not wanted (K >= 2 only)
  AGCN_REQUIRE(d_dX || !m.full, "backward: d_dX is required with metric_grad = full");
  if (need_G) {  // G_k = dYpre W_k^T   (K == 1: this is dX); W_k^T was split by the forward pass
    GemmArgs g = g_gemm_args(desc, R, dYp, d_weight, (K == 1) ? d_dX : wk.G);
    GemmArgs probe = g_gemm_args(desc, R, d_Y, d_weight, wk.G);
    const bool presplit = (desc->flags & AGCN_SAVE_FOR_BACKWARD) && tc_gemm_supported(probe);
    if ((rc = node_gemm(g, sv.tcG, st, presplit))) return rc;
  }
  GraphArgs ga;
  ga.plan = plan; ga.F = F; ga.K = K;
  ga.variant = desc->variant; ga.lap_mode = desc->laplacian_mode; ga.metric_full = m.full;
  ga.X = d_X; ga.XW = sv.XW; ga.Lint = d_Lint; ga.Lprev = has_prev ? d_Lprev : nullptr;
  ga.alpha = d_alpha; ga.beta = d_beta;
  ga.T = sv.T; ga.Lall = m.shortcut ? nullptr : sv.Lall;
  ga.dist = sv.dist; ga.dis = sv.dis; ga.stats = sv.stats;
  ga.G = wk.G; ga.dLall_in = d_dLall_in; ga.dX = dXbuf; ga.dL = wk.dL;
  ga.dl_parts = (m.need_dL && K >= 2) ? dl_parts(desc, plan) : 1;
  ga.dl_stride = dl_stride(plan);
  ga.dLprev = has_prev ? d_dLprev : nullptr;
  ga.dXW = wk.dXW; ga.dalpha_part = wk.dalpha_part; ga.dbeta_part = m.reslap ? wk.dbeta_part : nullptr;
  ga.big_work = wk.big;
  // dweight[f*K + k, :] = T_k^T dYpre
  {
    GemmTNArgs t;
    t.M = R; t.Kd = F; t.N = Fo; t.S = K;
    t.A0 = d_X; t.lda0 = F;
    t.A1 = sv.T; t.lda1 = F; t.sliceA1 = (int64_t)R * F;
    t.D = dYp; t.ldd = Fo;
    t.out = d_dweight; t.partial = wk.tn_part;
    if ((rc = node_gemm_tn(t, plan->side))) return rc;
  }
  AGCN_CUDA(cudaEventRecord(plan->ev_side_join, plan->side));
  if (vfirst) {
    const float* Lf = m.shortcut ? d_Lint : sv.Lall;
    const int ident = m.shortcut ? 1 : 0;
    const bool other = cheb_tiles_has_mid(plan);
    if (other) {
      AGCN_CUDA(cudaEventRecord(plan->ev_big_fork, st));
      AGCN_CUDA(cudaStreamWaitEvent(plan->big, plan->ev_big_fork, 0));
    }
    if ((rc = cheb_tiles_forward(plan, dYp, Lf, ident, Fo, K, wk.V, st, plan->big, /*transL=*/1))) return rc;
    if (other) {
      AGCN_CUDA(cudaEventRecord(plan->ev_big_join, plan->big));
      AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_big_join, 0));
    }
    if ((rc = pre_forward(plan, -1, 0, dYp, wk.V, sv.ftG, nullptr, AGCN_ACT_LINEAR, /*F=*/Fo, /*Fo=*/F, K, d_dX, st))) return rc;
  } else if (fuse_b) {
    // G_z = dYpre W_z^T over every packed row on the tensor cores (relu' applied to the operand rows as they are
    // loaded), then the reverse recurrences on the CUDA cores
    const float* Lf = m.shortcut ? d_Lint : sv.Lall;
    const int ident = m.shortcut ? 1 : 0;
    if ((rc = pre_backward(plan, -1, 0, d_dY, desc->activation == AGCN_ACT_RELU ? d_Y : nullptr, sv.ftG, F, Fo, K, wk.G, st)))
      return rc;
    const bool other = cheb_tiles_has_mid(plan) || plan->large_tiles > 0;
    if (other) {
      AGCN_CUDA(cudaEventRecord(plan->ev_big_fork, st));
      AGCN_CUDA(cudaStreamWaitEvent(plan->big, plan->ev_big_fork, 0));
    }
    if ((rc = cheb_tiles_backward(plan, wk.G, Lf, ident, F, K, d_dX, st, plan->big))) return rc;
    if (plan->large_tiles > 0 && (rc = graph_recurrence_bwd(ga, false, plan->big, AGCN_SMALL_MAX))) return rc;
    if (other) {
      AGCN_CUDA(cudaEventRecord(plan->ev_big_join, plan->big));
      AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_big_join, 0));
    }
  } else if (K >= 2) {
    if (need_G && (rc = graph_recurrence_bwd(ga, m.need_dL, st))) return rc;
  } else if (m.need_dL) {
    if (d_dLall_in)
      AGCN_CUDA(cudaMemcpyAsync(wk.dL, d_dLall_in, (size_t)plan->LL * sizeof(float), cudaMemcpyDeviceToDevice, st));
    else
      AGCN_CUDA(cudaMemsetAsync(wk.dL, 0, (size_t)plan->LL * sizeof(float), st));
  }
  AGCN_CUDA(cudaStreamWaitEvent(st, plan->ev_side_join, 0));
  if (m.need_dL) {
    if ((rc = graph_laplacian_bwd(ga, st))) return rc;
    if ((rc = reduce_scalar_parts(wk.dalpha_part, plan->B, d_dalpha, st))) return rc;
    if (m.reslap) {
      if ((rc = reduce_scalar_parts(wk.dbeta_part, plan->B, d_dbeta, st))) return rc;
    }
  } else {
    if ((rc = zero_async(d_dalpha, 1, st))) return rc;  // res_L == I >= 0: leaky never sees alpha
  }
  if (m.full) {
    GemmTNArgs t;  // dM_L = X^T dXW
    t.M = R; t.Kd = F; t.N = F; t.S = 1;
    t.A0 = d_X; t.lda0 = F;
    t.D = wk.dXW; t.ldd = F;
    t.out = d_dM_L; t.partial = wk.tn_part;
    if ((rc = node_gemm_tn(t, st))) return rc;
    GemmArgs g;  // dX += dXW M_L^T
    g.M = R; g.N = F; g.Kd = F;
    g.A0 = wk.dXW; g.lda0 = F;
    g.B = d_M_L; g.ldb = F; g.transB = 1;
    g.C = d_dX; g.ldc = F; g.accumulate = 1;
    if ((rc = node_gemm(g, wk.tcM, st))) return rc;
  } else {
    // tf.py_func has no gradient: M_L receives none (graphconv.py:211, SURVEY Q1)
    if ((rc = zero_async(d_dM_L, (size_t)F * F, st))) return rc;
  }
  return AGCN_OK;
}

}  // namespace

extern "C" {

/* Building block exported for tests and tuning: out[(f*S + s)*N + c] = sum_r A_s[r, f] * D[r, c].
 * use_tensor_cores = 0 forces the CUDA-core kernel.  scratch: agcn_gemm_tn_scratch_bytes() bytes. */
size_t agcn_gemm_tn_scratch_bytes(int32_t M, int32_t Kd, int32_t N, int32_t S) {
  GemmTNArgs t;
  t.M = M; t.Kd = Kd; t.N = N; t.S = S;
  return 4 * std::max(gemm_tn_partial_floats(M, Kd, N, S), tc_gemm_tn_partial_floats(t)) + 256;
}

int agcn_gemm_tn(const float* d_A0, const float* d_A1, const float* d_D, float* d_out, int32_t M, int32_t Kd,
                 int32_t N, int32_t S, void* d_scratch, int32_t use_tensor_cores, void* stream) {
  AGCN_REQUIRE(d_A0 && d_D && d_out && d_scratch && M >= 1 && Kd >= 1 && N >= 1 && S >= 1, "gemm_tn: bad arguments");
  GemmTNArgs t;
  t.M = M; t.Kd = Kd; t.N = N; t.S = S;
  t.A0 = d_A0; t.lda0 = Kd;
  t.A1 = d_A1; t.lda1 = Kd; t.sliceA1 = (int64_t)M * Kd;
  t.D = d_D; t.ldd = N;
  t.out = d_out; t.partial = reinterpret_cast<float*>(d_scratch);
  if (use_tensor_cores) {
    if (!tc_gemm_tn_supported(t)) {
      set_error("gemm_tn: shape not supported by the tensor-core kernel");
      return AGCN_ERR_INVALID;
    }
    return tc_gemm_tn(t, (cudaStream_t)stream);
  }
  return gemm_tn(t, (cudaStream_t)stream);
}

/* Node-level linear map over the packed rows, the building block of the layers around SGC-LL that are plain
 * per-graph matmuls in the reference (BlockEnd blockend.py:67-86, DenseBlockEnd densenet_block.py:98-131, MLP
 * MLP.py:69-83, DenseMol dense_layer.py:33-50): because the rows of all graphs are stored back to back, "for every
 * graph: x_g W" is ONE [R, Kd] x [Kd, N] product. */
size_t agcn_node_gemm_scratch_bytes(int32_t N, int32_t Kd) { return 4 * tc_gemm_scratch_floats(N, Kd, 1, 1) + 256; }

int agcn_node_gemm(const float* d_A, int32_t lda, const float* d_B, int32_t ldb, int32_t transB, float* d_C, int32_t ldc,
                   int32_t M, int32_t N, int32_t Kd, const float* d_bias, const float* d_scale, int32_t accumulate,
                   int32_t activation, void* d_scratch, void* stream) {
  AGCN_REQUIRE(d_A && d_B && d_C && d_scratch && M >= 1 && N >= 1 && Kd >= 1, "node_gemm: bad arguments");
  AGCN_REQUIRE(activation == AGCN_ACT_LINEAR || activation == AGCN_ACT_RELU, "node_gemm: unknown activation");
  GemmArgs g;
  g.M = M; g.N = N; g.Kd = Kd;
  g.A0 = d_A; g.lda0 = lda;
  g.B = d_B; g.ldb = ldb; g.transB = transB;
  g.C = d_C; g.ldc = ldc;
  g.bias = d_bias; g.scale = d_scale; g.accumulate = accumulate; g.act = activation;
  return node_gemm(g, reinterpret_cast<float*>(d_scratch), (cudaStream_t)stream);
}

/* bench.py's roofline: CUDA-event timing of the fused forward kernel on its launching stream */
int agcn_fused_profile(int enable) {
  fused_profile_enable(enable);
  return AGCN_OK;
}
int agcn_fused_profile_read(float* ms_sum, int* launches) { return fused_profile_read(ms_sum, launches); }

/* tuning aid: per-tile timeline (nanosecond stamps) of the fused forward kernel; NULL switches it off */
int agcn_fused_debug_set(void* d_buf) {
  fused_debug_set(d_buf);
  return AGCN_OK;
}

int agcn_sgcll_host_scratch_bytes(const agcn_sgcll_desc* desc, const agcn_plan* plan, size_t* bytes) {
  AGCN_REQUIRE(desc && plan && bytes, "null pointer");
  *bytes = carve_host(desc, plan, nullptr).bytes;
  return AGCN_OK;
}

int agcn_sgcll_forward_host(const agcn_sgcll_desc* desc, const agcn_plan* plan, const float* h_X_padded,
                            const float* h_L_padded, const float* d_M_L, const float* d_weight, const float* d_bias,
                            const float* d_alpha, float* h_Y_padded, void* d_scratch, size_t scratch_bytes,
                            void* stream) {
  int rc = check_desc(desc, plan);
  if (rc) return rc;
  AGCN_REQUIRE(h_X_padded && h_L_padded && h_Y_padded && d_scratch, "forward_host: null pointer");
  AGCN_REQUIRE(desc->variant == AGCN_VARIANT_SGC_LL, "forward_host: SGC_LL only");
  AGCN_REQUIRE((desc->flags & (AGCN_OUT_RES_L | AGCN_OUT_RES_W | AGCN_OUT_L_ALL)) == 0,
               "forward_host: optional outputs are not supported");
  const HostScratch h = carve_host(desc, plan, d_scratch);
  if (h.bytes > scratch_bytes) {
    set_error("forward_host: scratch too small");
    return AGCN_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const size_t B = plan->B, N = plan->Nmax;
  // Page-locked host arrays are mapped into the device's address space: the pack kernels then read them in place
  // and only the n_g real rows of every graph cross PCIe (the zero padding of the wire layout, 98 % of a
  // molecule batch, never moves).  Pageable arrays are staged through the copy engine.
  auto device_view = [](const float* h) -> const float* {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, h) != cudaSuccess) {
      (void)cudaGetLastError();
      return nullptr;
    }
    if ((at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged) && at.devicePointer)
      return reinterpret_cast<const float*>(at.devicePointer);
    return nullptr;
  };
  const float* xsrc = device_view(h_X_padded);
  const float* lsrc = device_view(h_L_padded);
  if (!xsrc) {
    AGCN_CUDA(cudaMemcpyAsync(h.Xpad, h_X_padded, B * N * desc->F * 4, cudaMemcpyHostToDevice, st));
    xsrc = h.Xpad;
  }
  if (!lsrc) {
    AGCN_CUDA(cudaMemcpyAsync(h.Lpad, h_L_padded, B * N * N * 4, cudaMemcpyHostToDevice, st));
    lsrc = h.Lpad;
  }
  if ((rc = agcn_pack_nodes(plan, xsrc, h.X, desc->F, st))) return rc;
  if ((rc = agcn_pack_lap(plan, lsrc, h.L, st))) return rc;
  if ((rc = agcn_sgcll_forward(desc, plan, h.X, h.L, nullptr, d_M_L, d_weight, d_bias, d_alpha, nullptr, h.Y, nullptr,
                               nullptr, nullptr, h.saved, h.work, h.work_bytes, st)))
    return rc;
  if ((rc = agcn_unpack_nodes(plan, h.Y, h.Ypad, desc->Fo, st))) return rc;
  AGCN_CUDA(cudaMemcpyAsync(h_Y_padded, h.Ypad, B * N * desc->Fo * 4, cudaMemcpyDeviceToHost, st));
  AGCN_CUDA(cudaStreamSynchronize(st));
  return AGCN_OK;
}

}  // extern "C"
