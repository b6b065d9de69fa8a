// Graph construction for point clouds on the device (SURVEY.md section 8f row 4): the threshold adjacency of the
// reference's loaders followed by Graph.compute_laplacian, for a whole packed batch.
//
//   rule MEAN    utils/data_loader/meshloader.py:264-285 (ModelNet40): d_lim = mean of ||p_i - p_j|| over the pairs
//                j <= i (the n zero self-distances included); i ~ j iff i != j and d_ij < d_lim
//   rule CUTOFF  utils/data_loader/pointcloudloader.py:240-263 (Sydney): d_lim = np.sort(all_dist)[-int(n * ratio)],
//                the int(n * ratio)-th LARGEST of the same distances (index -0 selects the smallest, a zero
//                self-distance: no edge at all)
//   Laplacian    models/graph_structure.py:85-130: A^ = D~^-1/2 (A + I) D~^-1/2, L = I - D^-1/2 A^ D^-1/2 with D from the
//                column sums of A^
//
// The reference runs this as O(n^2) interpreted Python per sample on the host; here every sweep is one warp per
// point over its row of the distance matrix, distances recomputed from the coordinates (F <= 8 floats per point) each
// time instead of stored: the only n x n traffic is the final write of L.  Degrees are exact integers, the two
// normalisations are evaluated in double (the reference's scipy path is float64), L is stored as float32 like the
// reference's feed (graph_topology.py:92-98).  The cut-off threshold is an exact order statistic (4-pass radix
// select over the float bit patterns, integer histograms: deterministic).
#include <algorithm>

#include "agcn_internal.cuh"

namespace agcn {
namespace pg {

constexpr int WARPS = 8;       // rows (points) per CTA
constexpr int MAXF = 8;

struct Args {
  const float* P;              // [R, F] packed points
  int F;
  const int32_t* n_nodes;
  const int32_t* node_off;
  const int64_t* lap_off;
  double* rowpart;             // [R]   mean rule: sum_{j<i} d_ij
  float* dlim;                 // [B]
  uint32_t* hist;              // [B][256]
  uint32_t* sel;               // [B][2] {prefix, k remaining}
  double* dinv;                // [R]   (deg + 1)^-1/2
  double* q;                   // [R]   second normalisation
  float* L;                    // packed out
  float ratio;
  int shift;                   // radix pass: byte at this bit offset
};

__device__ __forceinline__ float dist_to(const float pi[MAXF], const float* __restrict__ pj, int F) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < MAXF; ++c)
    if (c < F) {
      const float d = pi[c] - __ldg(pj + c);
      s = fmaf(d, d, s);
    }
  return sqrtf(s);
}

__device__ __forceinline__ bool row_setup(const Args& a, int& g, int& i, int& n, int& off, float pi[MAXF]) {
  g = blockIdx.y;
  i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  n = a.n_nodes[g];
  off = a.node_off[g];
  if (i >= n) return false;
#pragma unroll
  for (int c = 0; c < MAXF; ++c) pi[c] = (c < a.F) ? __ldg(a.P + (int64_t)(off + i) * a.F + c) : 0.f;
  return true;
}

// ---- MEAN rule
__global__ void __launch_bounds__(WARPS * 32) mean_rows_kernel(Args a) {
  int g, i, n, off;
  float pi[MAXF];
  if (!row_setup(a, g, i, n, off, pi)) return;
  const int lane = threadIdx.x & 31;
  double s = 0.0;
  for (int j = lane; j < i; j += 32) s += (double)dist_to(pi, a.P + (int64_t)(off + j) * a.F, a.F);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) a.rowpart[off + i] = s;
}

__global__ void __launch_bounds__(256) mean_reduce_kernel(Args a) {
  __shared__ double red[256];
  const int g = blockIdx.x, n = a.n_nodes[g], off = a.node_off[g];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) s += a.rowpart[off + i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) a.dlim[g] = (float)(red[0] / (0.5 * (double)n * (double)(n + 1)));
}

// ---- CUTOFF rule: radix select of the k-th largest key among the n (n + 1) / 2 distances of the pairs j <= i
__global__ void cut_init_kernel(Args a, int B) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= B) return;
  a.sel[2 * g] = 0u;
  a.sel[2 * g + 1] = (uint32_t)(int)((float)a.n_nodes[g] * a.ratio);   // int(n_p * sparse_ratio)
}

__global__ void __launch_bounds__(WARPS * 32) cut_hist_kernel(Args a) {
  __shared__ uint32_t sh[256];
  for (int b = threadIdx.x; b < 256; b += blockDim.x) sh[b] = 0u;
  __syncthreads();
  int g, i, n, off;
  float pi[MAXF];
  const bool live = row_setup(a, g, i, n, off, pi);
  if (live) {
    const int lane = threadIdx.x & 31;
    const uint32_t prefix = a.sel[2 * g];
    const int hs = a.shift + 8;   // bits above the current byte must match the prefix
    for (int j = lane; j <= i; j += 32) {
      const uint32_t key = (j == i) ? 0u : __float_as_uint(dist_to(pi, a.P + (int64_t)(off + j) * a.F, a.F));
      if (hs >= 32 || (key >> hs) == (prefix >> hs)) atomicAdd(&sh[(key >> a.shift) & 255u], 1u);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < 256; b += blockDim.x)
    if (sh[b]) atomicAdd(&a.hist[(int64_t)blockIdx.y * 256 + b], sh[b]);
}

__global__ void cut_select_kernel(Args a, int B, int last) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= B) return;
  uint32_t* h = a.hist + (int64_t)g * 256;
  uint32_t k = a.sel[2 * g + 1], prefix = a.sel[2 * g];
  if (k > 0) {
    uint32_t cum = 0;
    int b = 255;
    for (; b > 0; --b) {
      if (cum + h[b] >= k) break;
      cum += h[b];
    }
    k -= cum;
    prefix |= (uint32_t)b << a.shift;
  }
  for (int b = 0; b < 256; ++b) h[b] = 0u;
  a.sel[2 * g] = prefix;
  a.sel[2 * g + 1] = k;
  if (last) a.dlim[g] = (a.sel[2 * g + 1] == 0u && prefix == 0u) ? 0.f : __uint_as_float(prefix);
}

// ---- degrees, second normalisation, Laplacian
__global__ void __launch_bounds__(WARPS * 32) degree_kernel(Args a) {
  int g, i, n, off;
  float pi[MAXF];
  if (!row_setup(a, g, i, n, off, pi)) return;
  const int lane = threadIdx.x & 31;
  const float lim = a.dlim[g];
  int deg = 0;
  for (int j = lane; j < n; j += 32)
    if (j != i && dist_to(pi, a.P + (int64_t)(off + j) * a.F, a.F) < lim) ++deg;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) deg += __shfl_xor_sync(0xffffffffu, deg, o);
  if (lane == 0) a.dinv[off + i] = 1.0 / sqrt((double)(deg + 1));   // row sum of A + I (graph_structure.py:114-116)
}

__global__ void __launch_bounds__(WARPS * 32) rowsum_kernel(Args a) {
  int g, i, n, off;
  float pi[MAXF];
  if (!row_setup(a, g, i, n, off, pi)) return;
  const int lane = threadIdx.x & 31;
  const float lim = a.dlim[g];
  double s = 0.0;
  for (int j = lane; j < n; j += 32)
    if (j == i || dist_to(pi, a.P + (int64_t)(off + j) * a.F, a.F) < lim) s += a.dinv[off + j];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  // d = colsum(A^) + eps, d^-1/2 (graph_structure.py:93-102); A^ is symmetric, eps = 4.9e-324 vanishes next to d >= 1/n
  if (lane == 0) a.q[off + i] = 1.0 / sqrt(a.dinv[off + i] * s);
}

__global__ void __launch_bounds__(WARPS * 32) laplacian_kernel(Args a) {
  int g, i, n, off;
  float pi[MAXF];
  if (!row_setup(a, g, i, n, off, pi)) return;
  const int lane = threadIdx.x & 31;
  const float lim = a.dlim[g];
  const double ri = a.q[off + i] * a.dinv[off + i];
  float* __restrict__ row = a.L + a.lap_off[g] + (int64_t)i * n;
  for (int j = lane; j < n; j += 32) {
    double v = 0.0;
    if (j == i)
      v = 1.0 - ri * ri;
    else if (dist_to(pi, a.P + (int64_t)(off + j) * a.F, a.F) < lim)
      v = -ri * (a.q[off + j] * a.dinv[off + j]);
    row[j] = (float)v;
  }
}

struct Work {
  double *rowpart, *dinv, *q;
  float* dlim;
  uint32_t *hist, *sel;
  size_t bytes;
};

static Work carve(const agcn_plan* plan, void* base) {
  Arena c(base);
  Work w{};
  w.rowpart = c.take<double>(plan->R);
  w.dinv = c.take<double>(plan->R);
  w.q = c.take<double>(plan->R);
  w.dlim = c.take((size_t)plan->B);
  w.hist = c.take<uint32_t>((size_t)plan->B * 256);
  w.sel = c.take<uint32_t>((size_t)plan->B * 2);
  w.bytes = c.bytes;
  return w;
}

}  // namespace pg
}  // namespace agcn

using namespace agcn;

extern "C" {

int agcn_point_laplacian_workspace_bytes(const agcn_plan* plan, size_t* bytes) {
  AGCN_REQUIRE(plan && bytes, "point_laplacian_workspace_bytes: null pointer");
  *bytes = pg::carve(plan, nullptr).bytes + 256;
  return AGCN_OK;
}

int agcn_point_laplacian(const agcn_plan* plan, const float* d_points, int32_t F, int32_t rule, float sparse_ratio,
                         float* d_L, void* d_work, size_t work_bytes, void* stream) {
  AGCN_REQUIRE(plan && d_points && d_L && d_work, "point_laplacian: null pointer");
  AGCN_REQUIRE(F >= 1 && F <= pg::MAXF, "point_laplacian: 1 <= F <= 8 coordinates per point");
  AGCN_REQUIRE(rule == AGCN_ADJ_MEAN_DISTANCE || rule == AGCN_ADJ_CUTOFF, "point_laplacian: unknown rule");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = plan_use(plan, st);
  if (rc) return rc;
  pg::Work w = pg::carve(plan, d_work);
  if (w.bytes > work_bytes) {
    set_error("point_laplacian: workspace too small");
    return AGCN_ERR_WORKSPACE;
  }
  pg::Args a{};
  a.P = d_points; a.F = F;
  a.n_nodes = plan->d_n; a.node_off = plan->d_node_off; a.lap_off = plan->d_lap_off;
  a.rowpart = w.rowpart; a.dlim = w.dlim; a.hist = w.hist; a.sel = w.sel; a.dinv = w.dinv; a.q = w.q;
  a.L = d_L; a.ratio = sparse_ratio; a.shift = 0;
  const int B = plan->B;
  const dim3 grid((plan->max_n + pg::WARPS - 1) / pg::WARPS, B);
  const int threads = pg::WARPS * 32;
  if (rule == AGCN_ADJ_MEAN_DISTANCE) {
    pg::mean_rows_kernel<<<grid, threads, 0, st>>>(a);
    AGCN_LAUNCH_CHECK();
    pg::mean_reduce_kernel<<<B, 256, 0, st>>>(a);
    AGCN_LAUNCH_CHECK();
  } else {
    AGCN_CUDA(cudaMemsetAsync(w.hist, 0, (size_t)B * 256 * 4, st));
    pg::cut_init_kernel<<<(B + 127) / 128, 128, 0, st>>>(a, B);
    AGCN_LAUNCH_CHECK();
    for (int pass = 0; pass < 4; ++pass) {
      a.shift = 24 - 8 * pass;
      pg::cut_hist_kernel<<<grid, threads, 0, st>>>(a);
      AGCN_LAUNCH_CHECK();
      pg::cut_select_kernel<<<(B + 127) / 128, 128, 0, st>>>(a, B, pass == 3);
      AGCN_LAUNCH_CHECK();
    }
  }
  pg::degree_kernel<<<grid, threads, 0, st>>>(a);
  AGCN_LAUNCH_CHECK();
  pg::rowsum_kernel<<<grid, threads, 0, st>>>(a);
  AGCN_LAUNCH_CHECK();
  {
    ProfScope prof("pg::laplacian_kernel", st);
    pg::laplacian_kernel<<<grid, threads, 0, st>>>(a);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // extern "C"
