// Node-level dense contractions of the SGC-LL layer: they run over ALL R = sum n_g nodes of the
// batch at once (no per-graph structure), fp32 with fp32 accumulation on the CUDA cores.
//
//   gemm_rows  : Y = act(sum_k T_k W_k + b)      graphconv.py:238-247 (stack/transpose/reshape/matmul)
//                XW = X M_L                       graphconv.py:164
//                G_k = dY W_k^T, dX += dXW M_L^T  (backward of the above)
//   gemm_tn    : dW_k = T_k^T dY, dM_L = X^T dXW  contraction over the node dimension, deterministic
//                two-stage reduction (no atomics)
//   act_bwd_colsum : dYpre = dY * relu'(Y) and dbias = colsum(dYpre)
//
// gemm_auto / gemm_tn_auto pick between these kernels and their tcgen05 versions (agcn_tc_gemm.cu) for every caller.
#include <algorithm>

#include "agcn_internal.cuh"

namespace agcn {

constexpr int BM = 64, BN = 64, BK = 16, PK = BK + 4;

// 256 threads, 4x4 outputs per thread.
template <bool VEC, bool TB>
__global__ void __launch_bounds__(256) gemm_rows_kernel(GemmArgs p) {
  __shared__ __align__(16) float As[BM][PK];
  __shared__ __align__(16) float Bs[BK][BN + 4];  // always [k][col]; B^T tiles are transposed on the way in
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN, z = blockIdx.z;
  float acc[4][4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int t = 0; t < 4; ++t) acc[q][t] = 0.f;

  for (int s = 0; s < p.S; ++s) {
    const float* __restrict__ A = (s == 0) ? p.A0 : p.A1 + (int64_t)(s - 1) * p.sliceA1;
    const int lda = (s == 0) ? p.lda0 : p.lda1;
    const float* __restrict__ Bm = p.B + (int64_t)(z * p.S + s) * p.sliceB;
    for (int k0 = 0; k0 < p.Kd; k0 += BK) {
      // ---- A tile [BM x BK]
      if (VEC) {
        const int row = tid >> 2, k4 = (tid & 3) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        const int m = m0 + row, k = k0 + k4;
        if (m < p.M && k < p.Kd) v = *reinterpret_cast<const float4*>(A + (int64_t)m * lda + k);  // Kd % 4 == 0
        *reinterpret_cast<float4*>(&As[row][k4]) = v;
      } else {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = tid + 256 * u, row = e / BK, kk = e % BK;
          const int m = m0 + row, k = k0 + kk;
          As[row][kk] = (m < p.M && k < p.Kd) ? A[(int64_t)m * lda + k] : 0.f;
        }
      }
      // ---- B tile
      if (!TB) {
        if (VEC) {
          const int kk = tid >> 4, c4 = (tid & 15) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          const int k = k0 + kk, c = n0 + c4;
          if (k < p.Kd && c < p.N) v = *reinterpret_cast<const float4*>(Bm + (int64_t)k * p.ldb + c);  // N % 4 == 0
          *reinterpret_cast<float4*>(&Bs[kk][c4]) = v;
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = tid + 256 * u, kk = e / BN, cc = e % BN;
            const int k = k0 + kk, c = n0 + cc;
            Bs[kk][cc] = (k < p.Kd && c < p.N) ? Bm[(int64_t)k * p.ldb + c] : 0.f;
          }
        }
      } else {
        if (VEC) {
          const int col = tid >> 2, k4 = (tid & 3) * 4;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          const int c = n0 + col, k = k0 + k4;
          if (c < p.N && k < p.Kd) v = *reinterpret_cast<const float4*>(Bm + (int64_t)c * p.ldb + k);
          Bs[k4 + 0][col] = v.x; Bs[k4 + 1][col] = v.y; Bs[k4 + 2][col] = v.z; Bs[k4 + 3][col] = v.w;
        } else {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = tid + 256 * u, col = e / BK, kk = e % BK;
            const int c = n0 + col, k = k0 + kk;
            Bs[kk][col] = (c < p.N && k < p.Kd) ? Bm[(int64_t)c * p.ldb + k] : 0.f;
          }
        }
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < BK; kk += 4) {
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
  }
  // ---- epilogue
  float* __restrict__ C = p.C + (int64_t)z * p.sliceC;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int m = m0 + ty * 4 + q;
    if (m >= p.M) continue;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int c = n0 + tx * 4 + t;
      if (c >= p.N) continue;
      float v = acc[q][t];
      if (p.scale) v *= __ldg(p.scale);
      if (p.bias) v += p.bias[c];
      if (p.accumulate) v += C[(int64_t)m * p.ldc + c];
      if (p.act == AGCN_ACT_RELU) v = fmaxf(v, 0.f);
      C[(int64_t)m * p.ldc + c] = v;
    }
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int gemm_rows(const GemmArgs& a, cudaStream_t st) {
  if (a.M <= 0 || a.N <= 0) return AGCN_OK;
  AGCN_REQUIRE(a.A0 && a.B && a.C && a.Kd > 0 && a.S >= 1 && a.Z >= 1, "gemm_rows: bad arguments");
  AGCN_REQUIRE(a.S == 1 || a.A1, "gemm_rows: A1 missing");
  bool vec = (a.Kd % 4 == 0) && (a.lda0 % 4 == 0) && aligned16(a.A0) && (a.ldb % 4 == 0) && aligned16(a.B) &&
             (a.sliceB % 4 == 0);
  if (a.S > 1) vec = vec && (a.lda1 % 4 == 0) && aligned16(a.A1) && (a.sliceA1 % 4 == 0);
  if (!a.transB) vec = vec && (a.N % 4 == 0);
  dim3 grid((a.M + BM - 1) / BM, (a.N + BN - 1) / BN, a.Z);
  if (vec) {
    if (a.transB)
      {
        ProfScope prof("gemm_rows_kernel", st);
        gemm_rows_kernel<true, true><<<grid, 256, 0, st>>>(a);
      }
    else
      {
        ProfScope prof("gemm_rows_kernel", st);
        gemm_rows_kernel<true, false><<<grid, 256, 0, st>>>(a);
      }
  } else {
    if (a.transB)
      {
        ProfScope prof("gemm_rows_kernel", st);
        gemm_rows_kernel<false, true><<<grid, 256, 0, st>>>(a);
      }
    else
      {
        ProfScope prof("gemm_rows_kernel", st);
        gemm_rows_kernel<false, false><<<grid, 256, 0, st>>>(a);
      }
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// ------------------------------------------------------------------------------------------------
// TN contraction over the node rows: split the rows over gridDim.x CTAs, each writes a partial
// [S][Kd][N] block; a second kernel sums the partials in a fixed order (deterministic).
constexpr int TN_ROWS = 16;  // rows staged per step

__global__ void __launch_bounds__(256) gemm_tn_kernel(GemmTNArgs p, int rows_per_split, int tiles_n) {
  __shared__ __align__(16) float As[TN_ROWS][BM + 4];
  __shared__ __align__(16) float Ds[TN_ROWS][BN + 4];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int split = blockIdx.x;
  const int f0 = (blockIdx.y / tiles_n) * BM, c0 = (blockIdx.y % tiles_n) * BN;
  const int s = blockIdx.z;
  const float* __restrict__ A = (s == 0) ? p.A0 : p.A1 + (int64_t)(s - 1) * p.sliceA1;
  const int lda = (s == 0) ? p.lda0 : p.lda1;
  const int r_begin = split * rows_per_split;
  const int r_end = min(p.M, r_begin + rows_per_split);
  float acc[4][4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int t = 0; t < 4; ++t) acc[q][t] = 0.f;
  for (int r0 = r_begin; r0 < r_end; r0 += TN_ROWS) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int e = tid + 256 * u, rr = e / BM, cc = e % BM;
      const int r = r0 + rr;
      const int f = f0 + cc, c = c0 + cc;
      As[rr][cc] = (r < r_end && f < p.Kd) ? A[(int64_t)r * lda + f] : 0.f;
      Ds[rr][cc] = (r < r_end && c < p.N) ? p.D[(int64_t)r * p.ldd + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < TN_ROWS; ++rr) {
      const float4 a = *reinterpret_cast<const float4*>(&As[rr][ty * 4]);
      const float4 d = *reinterpret_cast<const float4*>(&Ds[rr][tx * 4]);
      acc[0][0] += a.x * d.x; acc[0][1] += a.x * d.y; acc[0][2] += a.x * d.z; acc[0][3] += a.x * d.w;
      acc[1][0] += a.y * d.x; acc[1][1] += a.y * d.y; acc[1][2] += a.y * d.z; acc[1][3] += a.y * d.w;
      acc[2][0] += a.z * d.x; acc[2][1] += a.z * d.y; acc[2][2] += a.z * d.z; acc[2][3] += a.z * d.w;
      acc[3][0] += a.w * d.x; acc[3][1] += a.w * d.y; acc[3][2] += a.w * d.z; acc[3][3] += a.w * d.w;
    }
    __syncthreads();
  }
  // partial layout: [split][(f*S + s)*N + c]
  float* __restrict__ P = p.partial + (int64_t)split * p.Kd * p.S * p.N;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int f = f0 + ty * 4 + q;
    if (f >= p.Kd) continue;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int c = c0 + tx * 4 + t;
      if (c < p.N) P[((int64_t)f * p.S + s) * p.N + c] = acc[q][t];
    }
  }
}

__global__ void reduce_partials_kernel(const float* __restrict__ partial, float* __restrict__ out, int64_t elems,
                                       int splits) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += partial[(int64_t)k * elems + e];
  out[e] = s;
}

static int tn_splits(int M, int Kd, int N, int S) {
  const int tiles = ((Kd + BM - 1) / BM) * ((N + BN - 1) / BN) * S;
  int splits = (4 * 148 + tiles - 1) / tiles;
  const int max_splits = (M + 63) / 64;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  return splits;
}

size_t gemm_tn_partial_floats(int M, int Kd, int N, int S) {
  return (size_t)tn_splits(M, Kd, N, S) * Kd * S * N;
}

int gemm_tn(const GemmTNArgs& a, cudaStream_t st) {
  AGCN_REQUIRE(a.A0 && a.D && a.out && a.partial && a.Kd > 0 && a.N > 0 && a.S >= 1, "gemm_tn: bad arguments");
  const int64_t elems = (int64_t)a.Kd * a.S * a.N;
  if (a.M <= 0) {
    AGCN_CUDA(cudaMemsetAsync(a.out, 0, elems * sizeof(float), st));
    return AGCN_OK;
  }
  const int splits = tn_splits(a.M, a.Kd, a.N, a.S);
  int rows_per_split = (a.M + splits - 1) / splits;
  rows_per_split = (rows_per_split + TN_ROWS - 1) / TN_ROWS * TN_ROWS;
  const int tiles_n = (a.N + BN - 1) / BN;
  dim3 grid(splits, ((a.Kd + BM - 1) / BM) * tiles_n, a.S);
  gemm_tn_kernel<<<grid, 256, 0, st>>>(a, rows_per_split, tiles_n);
  AGCN_LAUNCH_CHECK();
  reduce_partials_kernel<<<(unsigned)((elems + 255) / 256), 256, 0, st>>>(a.partial, a.out, elems, splits);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// ------------------------------------------------------------------------------------------------
// Engine of every node-level product: tensor cores when the operands are TMA-compatible, CUDA cores otherwise (F = 75)
int gemm_auto(const GemmArgs& a, float* tc_scratch, cudaStream_t st, bool presplit) {
  if (!tc_gemm_supported(a)) return gemm_rows(a, st);
  if (!presplit) {
    int rc = tc_gemm_split_b(a, tc_scratch, st);
    if (rc) return rc;
  }
  return tc_gemm(a, tc_scratch, st);
}

int gemm_tn_auto(const GemmTNArgs& a, cudaStream_t st) {
  return tc_gemm_tn_supported(a) ? tc_gemm_tn(a, st) : gemm_tn(a, st);
}

size_t gemm_tn_auto_partial_floats(const GemmTNArgs& a) {
  return std::max(tc_gemm_tn_partial_floats(a), gemm_tn_partial_floats(a.M, a.Kd, a.N, a.S));
}

// ------------------------------------------------------------------------------------------------
constexpr int ACT_ROWS = 64;  // rows per CTA

// dYp = dY * relu'(Y); per-CTA column sums.  Threads are laid out [row lane][column]: consecutive threads
// walk consecutive columns (coalesced), the row lanes of a column are combined through shared memory.
__global__ void __launch_bounds__(256) act_bwd_colsum_kernel(const float* __restrict__ dY, const float* __restrict__ Y,
                                                             float* __restrict__ dYp, float* __restrict__ partial,
                                                             int64_t R, int Fo, int act) {
  __shared__ float red[256];
  const int64_t r0 = (int64_t)blockIdx.x * ACT_ROWS;
  const int64_t r1 = min(R, r0 + ACT_ROWS);
  const int cols = min(Fo, 256);             // columns handled per pass
  const int lanes = 256 / cols > 0 ? 256 / cols : 1;  // row lanes per column
  for (int cbase = 0; cbase < Fo; cbase += cols) {
    const int c = cbase + (int)(threadIdx.x % cols), rl = threadIdx.x / cols;
    float s = 0.f;
    if (c < Fo && rl < lanes) {
      for (int64_t r = r0 + rl; r < r1; r += lanes) {
        float g = dY[r * Fo + c];
        if (act == AGCN_ACT_RELU) {
          g = (Y[r * Fo + c] > 0.f) ? g : 0.f;
          dYp[r * Fo + c] = g;
        }
        s += g;
      }
    }
    red[threadIdx.x] = s;
    __syncthreads();
    if (rl == 0 && c < Fo) {
      for (int l = 1; l < lanes; ++l) s += red[l * cols + (threadIdx.x % cols)];
      partial[(int64_t)blockIdx.x * Fo + c] = s;
    }
    __syncthreads();
  }
}

// out[c] = sum_k partial[k][c]: 32 columns per CTA, the k range split over 8 warps, fixed summation order
__global__ void __launch_bounds__(256) colsum_reduce_kernel(const float* __restrict__ partial, float* __restrict__ out,
                                                            int n_part, int Fo) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < Fo)
    for (int k = w; k < n_part; k += 8) s += partial[(int64_t)k * Fo + c];
  red[w][lane] = s;
  __syncthreads();
  if (w == 0 && c < Fo) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][lane];
    out[c] = t;
  }
}

size_t act_bwd_partial_floats(int64_t R, int Fo) { return (size_t)((R + ACT_ROWS - 1) / ACT_ROWS) * Fo; }

// stage 1 (stream st): dYp and the per-CTA column sums; stage 2 (stream st2, ordered after stage 1 by the
// caller): dbias.  Split so that the reduction can leave the critical path of the backward pass.
int act_bwd_partials(const float* dY, const float* Y, float* dYp, float* partial, int64_t R, int Fo, int act,
                     cudaStream_t st) {
  if (R <= 0) return AGCN_OK;
  const int blocks = (int)((R + ACT_ROWS - 1) / ACT_ROWS);
  act_bwd_colsum_kernel<<<blocks, 256, 0, st>>>(dY, Y, dYp, partial, R, Fo, act);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

int act_bwd_reduce(const float* partial, float* dbias, int64_t R, int Fo, cudaStream_t st) {
  if (R <= 0) {
    AGCN_CUDA(cudaMemsetAsync(dbias, 0, Fo * sizeof(float), st));
    return AGCN_OK;
  }
  return colsum_reduce(partial, (int)((R + ACT_ROWS - 1) / ACT_ROWS), Fo, dbias, st);
}

int colsum_reduce(const float* partial, int n_part, int cols, float* out, cudaStream_t st) {
  colsum_reduce_kernel<<<(cols + 31) / 32, 256, 0, st>>>(partial, out, n_part, cols);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // namespace agcn
