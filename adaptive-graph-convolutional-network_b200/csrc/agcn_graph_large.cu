// Row-tiled path for graphs with more than AGCN_SMALL_MAX nodes (point clouds: ModelNet40-shape
// N = 1024, Sydney-shape ragged N, the N <= 4096 sweep): the n x n Laplacian does not fit in shared
// memory, so every Chebyshev step is a grouped GEMM over (graph, 64-row tile) work items,
//     Out = cmul * op(L_g) * In  (+ Add)  (- Sub),        op(L) = L + I | L | L^T (+ I)
// with L streamed from HBM/L2 in 64 x 16 tiles.  Forward: graphconv.py:221-236; backward: its
// reverse recurrence (see agcn_graph_small.cu).
#include "agcn_internal.cuh"

namespace agcn {

constexpr int GM = 64, GN = 64, GK = 16;

__global__ void __launch_bounds__(256) grouped_lap_gemm_kernel(GroupedArgs p) {
  __shared__ __align__(16) float As[GM][GK + 4];
  __shared__ __align__(16) float Bs[GK][GN + 4];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int g = p.tile_graph[blockIdx.x], m0 = p.tile_row[blockIdx.x];
  const int n = p.n_nodes[g];
  const int64_t row0 = p.node_off[g];
  const float* __restrict__ Lg = p.L + p.lap_off[g];
  const int c0 = blockIdx.y * GN;
  float acc[4][4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int t = 0; t < 4; ++t) acc[q][t] = 0.f;
  // register-staged double buffering: the global loads of tile k+1 are in flight while tile k is multiplied
  float ra[4], rb[4];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = tid + 256 * u;
      int row, kk;
      if (!p.transL) {
        row = e / GK; kk = e % GK;
      } else {
        kk = e / GM; row = e % GM;  // consecutive threads walk a row of L
      }
      const int i = m0 + row, j = k0 + kk;
      float v = 0.f;
      if (i < n && j < n) {
        v = p.transL ? Lg[(int64_t)j * n + i] : Lg[(int64_t)i * n + j];
        if (p.add_identity && i == j) v += 1.f;
      }
      ra[u] = v;
      const int bk = e / GN, cc = e % GN;
      const int jj = k0 + bk, c = c0 + cc;
      rb[u] = (jj < n && c < p.F) ? p.In[(row0 + jj) * p.F + c] : 0.f;
    }
  };
  auto stash = [&]() {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = tid + 256 * u;
      if (!p.transL)
        As[e / GK][e % GK] = ra[u];
      else
        As[e % GM][e / GM] = ra[u];
      Bs[e / GN][e % GN] = rb[u];
    }
  };
  fetch(0);
  for (int k0 = 0; k0 < n; k0 += GK) {
    stash();
    __syncthreads();
    if (k0 + GK < n) fetch(k0 + GK);
#pragma unroll
    for (int kk = 0; kk < GK; kk += 4) {
      float4 a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) a[q] = *reinterpret_cast<const float4*>(&As[ty * 4 + q][kk]);
#pragma unroll
      for (int u = 0; u < 4; ++u) b[u] = *reinterpret_cast<const float4*>(&Bs[kk + u][tx * 4]);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        acc[q][0] += a[q].x * b[0].x + a[q].y * b[1].x + a[q].z * b[2].x + a[q].w * b[3].x;
        acc[q][1] += a[q].x * b[0].y + a[q].y * b[1].y + a[q].z * b[2].y + a[q].w * b[3].y;
        acc[q][2] += a[q].x * b[0].z + a[q].y * b[1].z + a[q].z * b[2].z + a[q].w * b[3].z;
        acc[q][3] += a[q].x * b[0].w + a[q].y * b[1].w + a[q].z * b[2].w + a[q].w * b[3].w;
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int i = m0 + ty * 4 + q;
    if (i >= n) continue;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int c = c0 + tx * 4 + t;
      if (c >= p.F) continue;
      const int64_t o = (row0 + i) * p.F + c;
      float v = p.cmul * acc[q][t];
      if (p.Add) v += p.Add[o];
      if (p.Sub) v -= p.Sub[o];
      if (p.RowScale) v += p.RowScale[row0 + i] * p.ScaleIn[o];
      p.Out[o] = v;
      if (p.Out2) p.Out2[o] = v;
    }
  }
}

int grouped_simt(int tiles, const GroupedArgs& g, cudaStream_t st) {
  dim3 grid(tiles, (g.F + GN - 1) / GN);
  {
    ProfScope prof("grouped_lap_gemm_kernel", st);
    grouped_lap_gemm_kernel<<<grid, 256, 0, st>>>(g);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// One Chebyshev-shaped product over the first `tiles` row tiles of the plan: tensor cores when the shape allows
// (agcn_big_tc.cu), a streaming kernel for the 3/4-feature first layers of point clouds, else the SIMT kernel above.
int grouped_launch(const agcn_plan* plan, int tiles, const GroupedArgs& g, cudaStream_t st) {
  if (tiles <= 0) return AGCN_OK;
  if (grouped_thin_supported(g)) return grouped_thin(tiles, g, st);
  if (grouped_tc_supported(g)) return grouped_tc(plan, tiles, g, st);
  return grouped_simt(tiles, g, st);
}

static GroupedArgs base_args(const agcn_plan* plan) {
  GroupedArgs k{};
  k.n_nodes = plan->d_n;
  k.node_off = plan->d_node_off;
  k.lap_off = plan->d_lap_off;
  k.tile_graph = plan->d_tile_graph;
  k.tile_row = plan->d_tile_row;
  return k;
}

int large_chebyshev_fwd(const GraphArgs& a, cudaStream_t st) {
  const agcn_plan* plan = a.plan;
  if (plan->large_tiles == 0 || a.K <= 1) return AGCN_OK;
  const bool shortcut = (a.Lall == nullptr);
  const int64_t slice = (int64_t)plan->R * a.F;
  for (int k = 1; k < a.K; ++k) {
    GroupedArgs g = base_args(plan);
    g.L = shortcut ? a.Lint : a.Lall;
    g.add_identity = shortcut ? 1 : 0;
    g.transL = 0;
    g.In = (k == 1) ? a.X : a.T + (int64_t)(k - 2) * slice;
    g.Sub = (k >= 2) ? ((k == 2) ? a.X : a.T + (int64_t)(k - 3) * slice) : nullptr;
    g.Add = nullptr;
    g.Out = a.T + (int64_t)(k - 1) * slice;
    g.Out2 = nullptr;
    g.cmul = (k == 1) ? 1.f : 2.f;
    g.F = a.F;
    if (int rc = grouped_launch(plan, plan->large_tiles, g, st)) return rc;
  }
  return AGCN_OK;
}

// U_j overwrites G_j in place (slice j of a.G); dX receives U_0.  big_only: only the graphs with
// n > AGCN_SMALL_MAX (the others accumulate dL in shared memory inside recur_bwd_kernel).
int large_recurrence_bwd(const GraphArgs& a, float* G, bool big_only, cudaStream_t st) {
  const agcn_plan* plan = a.plan;
  const int tiles = big_only ? plan->big_tiles : plan->large_tiles;
  if (tiles == 0 || a.K <= 1) return AGCN_OK;
  const bool shortcut = (a.Lall == nullptr);
  const int64_t slice = (int64_t)plan->R * a.F;
  for (int j = a.K - 2; j >= 0; --j) {
    GroupedArgs g = base_args(plan);
    g.L = shortcut ? a.Lint : a.Lall;
    g.add_identity = shortcut ? 1 : 0;
    g.transL = 1;
    g.In = G + (int64_t)(j + 1) * slice;
    g.Add = G + (int64_t)j * slice;
    g.Sub = (j + 2 <= a.K - 1) ? G + (int64_t)(j + 2) * slice : nullptr;
    g.Out = G + (int64_t)j * slice;
    g.Out2 = (j == 0) ? a.dX : nullptr;
    g.cmul = (j + 1 >= 2) ? 2.f : 1.f;
    g.F = a.F;
    if (int rc = grouped_launch(plan, tiles, g, st)) return rc;
  }
  return AGCN_OK;
}

// Out[rows of the first `tiles` tiles] = cmul * M_g In + row_scale[row] * scale_in[row, :]
int grouped_rows_gemm(const agcn_plan* plan, int tiles, const float* Lmat, const float* In, float cmul,
                      const float* row_scale, const float* scale_in, float* Out, int F, cudaStream_t st) {
  if (tiles == 0) return AGCN_OK;
  GroupedArgs g = base_args(plan);
  g.L = Lmat; g.add_identity = 0; g.transL = 0;
  g.In = In; g.Sub = nullptr; g.Add = nullptr;
  g.Out = Out; g.Out2 = nullptr; g.cmul = cmul; g.F = F;
  g.RowScale = row_scale; g.ScaleIn = scale_in;
  return grouped_launch(plan, tiles, g, st);
}

}  // namespace agcn

// Tuning / debugging aid (include/agcn_sgcll.h): one row-tiled product over every graph above cheb_small_max,
// impl 0 = dispatcher, 1 = SIMT, 2 = tensor cores, 3 = thin.
extern "C" int agcn_debug_grouped_product(const agcn_plan* plan, const float* d_L, const float* d_In, float* d_Out,
                                          int32_t F, int32_t transL, int32_t add_identity, float cmul, int32_t impl,
                                          void* stream) {
  using namespace agcn;
  AGCN_REQUIRE(plan && d_L && d_In && d_Out && F >= 1, "null pointer or F < 1");
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = plan_use(plan, st)) return rc;
  GroupedArgs g = base_args(plan);
  g.L = d_L; g.add_identity = add_identity; g.transL = transL;
  g.In = d_In; g.Sub = nullptr; g.Add = nullptr; g.Out = d_Out; g.Out2 = nullptr; g.cmul = cmul; g.F = F;
  const int tiles = plan->large_tiles;
  if (tiles == 0) return AGCN_OK;
  switch (impl) {
    case 1: return grouped_simt(tiles, g, st);
    case 2: return grouped_tc(plan, tiles, g, st);
    case 4:   // the equal-size-graph kernel whatever the grid size (errors out when the batch is not eligible)
      g.force_uniform = 1;
      AGCN_REQUIRE(plan->uniform_n > 0 && plan->uniform_n % 128 == 0 && grouped_tc_supported(g),
                   "debug_grouped_product: impl 4 needs equal-size graphs with n % 128 == 0");
      return grouped_tc(plan, tiles, g, st);
    case 3: return grouped_thin(tiles, g, st);
    default: return grouped_launch(plan, tiles, g, st);
  }
}

