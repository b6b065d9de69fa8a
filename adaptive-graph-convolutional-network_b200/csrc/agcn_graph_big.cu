// Laplacian construction and its gradient for "big" graphs (n > AGCN_SMALL_MAX: point clouds such as the
// ModelNet40-shape N = 1024, the ragged Sydney shape, the N <= 4096 sweep).  The n x n matrices of such a
// graph do not fit in shared memory, so the chain of graphconv.py:163-216 / graphconv_reslap.py:136-195 is
// split into sweeps over (graph, 64-row tile) work items with the whole-matrix reductions (row sums of the
// similarity, Frobenius norms of the clips) carried between sweeps as per-tile partials that are summed in a
// fixed order (deterministic, no atomics):
//
//   forward   pair<SIM>   dist_ij = |xw_i - xw_j| by direct differences, W = exp(-dist), row-sum partials
//             dis         d^-1/2                                              graphconv.py:195-197
//             sweep<NORM> sum R^2 (and, Reslap, the quadratic forms of the second clip)   :212 / reslap :185,194
//             stats       s1, s2 per graph
//             sweep<FINAL> res_L, L_all                                       :213-216 / reslap :186-195
//   backward  pair<DL>    dL = dLall_in + sum_k c_k U_k T_{k-1}^T             (reverse of :221-236)
//             sweep<B1>, sweep<B2>  clip / leaky / sum chain -> d alpha, d beta, d L_prev
//             trans<B3>, trans<B4>  metric block (metric_grad = full): d(d^-1/2), C = d dist / dist
//             grouped GEMM          dXW = rowsum(C) xw - C XW
#include "agcn_internal.cuh"

namespace agcn {

namespace {

struct BigPtrs {
  const int32_t* n_nodes;
  const int32_t* node_off;
  const int32_t* order;
  const int32_t* tile_graph;
  const int32_t* tile_row;
  const int32_t* big_tile_start;
  const int64_t* lap_off;
};

BigPtrs big_ptrs(const agcn_plan* p) {
  return BigPtrs{p->d_n, p->d_node_off, p->d_order, p->d_tile_graph, p->d_tile_row, p->d_big_tile_start, p->d_lap_off};
}

__device__ __forceinline__ float leaky(float x, float alpha) { return fmaxf(x, 0.f) - alpha * fmaxf(-x, 0.f); }
__device__ __forceinline__ float leaky_grad(float x, float alpha) { return x > 0.f ? 1.f : (x < 0.f ? alpha : 0.f); }

// all 256 threads call; result valid in thread 0
template <int NV>
__device__ __forceinline__ void block_sum_vec(float (&v)[NV], float* red /* >= 8*NV floats */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
  }
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) red[wid * NV + k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      float s = 0.f;
      for (int w = 0; w < 8; ++w) s += red[w * NV + k];
      v[k] = s;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// pair kernel: 64 x 64 tile of an n x n matrix built from two row panels of node matrices
// ------------------------------------------------------------------------------------------------
constexpr int PT = 64, PK = 16;
enum { PAIR_SIM = 0, PAIR_DL = 1 };

struct PairArgs {
  BigPtrs pp;
  int F;
  // PAIR_SIM
  const float* XW;
  float* dist;
  float* resW;
  float* rowpart;  // [R][ncb]
  int ncb;
  // PAIR_DL
  int S;           // K - 1
  const float* U;  // U_k = slice k of the G buffer
  const float* X;  // T_0
  const float* T;  // T_1 .. T_{K-1}
  int64_t slice;
  const float* dL_in;
  float* dL;
};

template <int MODE>
__global__ void __launch_bounds__(256) big_pair_kernel(PairArgs p) {
  __shared__ __align__(16) float As[PK][PT + 4];
  __shared__ __align__(16) float Bs[PK][PT + 4];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int g = p.pp.tile_graph[blockIdx.x], m0 = p.pp.tile_row[blockIdx.x];
  const int n = p.pp.n_nodes[g];
  const int j0 = blockIdx.y * PT;
  if (j0 >= n) return;
  const int64_t row0 = p.pp.node_off[g];
  const int64_t loff = p.pp.lap_off[g];
  float acc[4][4];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[q][u] = 0.f;
  const int S = (MODE == PAIR_SIM) ? 1 : p.S;
  for (int s = 0; s < S; ++s) {
    const float* __restrict__ A = (MODE == PAIR_SIM) ? p.XW : p.U + (int64_t)(s + 1) * p.slice;
    const float* __restrict__ Bm = (MODE == PAIR_SIM) ? p.XW : (s == 0 ? p.X : p.T + (int64_t)(s - 1) * p.slice);
    const float coef = (MODE == PAIR_DL && s + 1 >= 2) ? 2.f : 1.f;  // c_1 = 1, c_k = 2
    for (int f0 = 0; f0 < p.F; f0 += PK) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = tid + 256 * u, row = e / PK, kk = e % PK;
        const int f = f0 + kk;
        const int i = m0 + row, j = j0 + row;
        As[kk][row] = (i < n && f < p.F) ? coef * A[(row0 + i) * p.F + f] : 0.f;
        Bs[kk][row] = (j < n && f < p.F) ? Bm[(row0 + j) * p.F + f] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < PK; ++kk) {
        const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (MODE == PAIR_SIM) {
              const float d = av[q] - bv[u];
              acc[q][u] += d * d;
            } else {
              acc[q][u] += av[q] * bv[u];
            }
          }
      }
      __syncthreads();
    }
  }
  if (MODE == PAIR_SIM) {
    // W_ij = exp(-dist), W_ii = 0 (graphconv.py:171-178); row sums of this 64-column block
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = m0 + ty * 4 + q;
      float rs = 0.f;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + tx * 4 + u;
        if (i < n && j < n) {
          const float d = sqrtf(acc[q][u]);
          const float w = (i == j) ? 0.f : expf(-d);
          const int64_t idx = loff + (int64_t)i * n + j;
          if (p.dist) p.dist[idx] = (i == j) ? 0.f : d;
          if (p.resW) p.resW[idx] = w;
          rs += w;
        }
      }
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);  // the 16 threads of one row
      if (tx == 0 && i < n && p.rowpart) p.rowpart[(row0 + i) * p.ncb + blockIdx.y] = rs;
    }
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = m0 + ty * 4 + q;
      if (i >= n) continue;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + tx * 4 + u;
        if (j >= n) continue;
        const int64_t idx = loff + (int64_t)i * n + j;
        p.dL[idx] = acc[q][u] + (p.dL_in ? p.dL_in[idx] : 0.f);
      }
    }
  }
}

// d = W.sum(axis=0) (W is symmetric), d^-1/2 with d == 0 -> 0 (graphconv.py:195-197, SURVEY Q8)
__global__ void big_dis_kernel(BigPtrs pp, const float* __restrict__ rowpart, int ncb, float* __restrict__ dis) {
  const int g = pp.tile_graph[blockIdx.x], m0 = pp.tile_row[blockIdx.x];
  const int n = pp.n_nodes[g];
  const int i = m0 + threadIdx.x;
  if (i >= n) return;
  const int64_t row = pp.node_off[g] + i;
  const int nb = (n + PT - 1) / PT;
  float d = 0.f;
  for (int c = 0; c < nb; ++c) d += rowpart[row * ncb + c];
  dis[row] = (d > AGCN_DEGREE_FLOOR) ? 1.0f / sqrtf(d) : 0.f;
}

// ------------------------------------------------------------------------------------------------
// elementwise sweeps over the rows of one tile (warp per row, lanes along the columns)
// ------------------------------------------------------------------------------------------------
enum { SW_NORM = 0, SW_FINAL = 1, SW_B1 = 2, SW_B2 = 3 };

struct SweepArgs {
  BigPtrs pp;
  int paper, reslap;
  const float* dist;
  const float* dis;
  const float* Lint;
  const float* Lprev;
  const float* alpha;
  const float* beta;
  const float* stats;  // [B][4] s1, s2, |R|^2, |Z|^2
  const float* gstat;  // [B][4] k2, k1 (backward)
  float* resL;
  float* Lall;
  float* Lall2;
  float* dL;
  float* dLprev;
  float* tilepart;  // [tiles][8]
};

// one element of a sweep: inputs by value, outputs through o* (written back by the caller when the pass stores them)
struct SweepCtx {
  float alpha, beta, s1, s2, k2;
  bool paper, reslap, has_prev, clipped2;
};

template <int PASS>
__device__ __forceinline__ void sweep_elem(const SweepCtx& c, bool diag, float dis_i, float dis_j, float dist, float lint,
                                           float lprev, float gd, float (&part)[4], float& o_resl, float& o_lall,
                                           float& o_dl, float& o_dlprev) {
  const float eye = diag ? 1.f : 0.f;
  float R = eye;
  if (c.paper) {
    const float w = diag ? 0.f : expf(-dist);
    R = eye - (dis_i * w) * dis_j;  // I - D^-1/2 W D^-1/2
  }
  if (PASS == SW_NORM) {
    part[0] += R * R;
    if (c.reslap) {
      const float lr = leaky(R, c.alpha);
      float cc = lint;
      if (c.has_prev) cc += lprev * c.beta;
      part[1] += lr * lr;
      part[2] += lr * cc;
      part[3] += cc * cc;
    }
    return;
  }
  const float u = R * c.s1;
  const float rl = leaky(u, c.alpha);    // graphconv.py:213
  float z = rl + lint;                   // graphconv.py:216
  if (c.has_prev) z += lprev * c.beta;   // graphconv_reslap.py:190
  if (PASS == SW_FINAL) {
    o_resl = rl;
    o_lall = c.reslap ? leaky(z * c.s2, c.alpha) : z;  // graphconv_reslap.py:194-195
  } else if (PASS == SW_B1) {
    // L_all = leaky(s2 Z): gradient w.r.t. v = s2 Z and <gv, Z>
    const float v = z * c.s2;
    part[0] -= gd * fmaxf(-v, 0.f);  // d alpha
    const float gv = gd * leaky_grad(v, c.alpha);
    part[1] += gv * z;
    o_dl = gv;
  } else {  // SW_B2
    float gz = gd;
    if (c.reslap && c.clipped2) gz = c.s2 * gz - z * c.k2;
    if (c.has_prev) {
      part[1] += gz * lprev;  // d beta
      o_dlprev = c.beta * gz;
    }
    part[0] -= gz * fmaxf(-u, 0.f);  // d alpha
    const float gu = gz * leaky_grad(u, c.alpha);
    part[2] += gu * R;
    o_dl = gu;
  }
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void stg4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }

// Which matrices a pass reads: a sweep is HBM-bound, so nothing is loaded that the pass does not use.
template <int PASS>
__global__ void __launch_bounds__(256) big_sweep_kernel(SweepArgs p) {
  __shared__ float red[8 * 4];
  const int t = blockIdx.x;
  const int g = p.pp.tile_graph[t], m0 = p.pp.tile_row[t];
  const int n = p.pp.n_nodes[g];
  const int64_t row0 = p.pp.node_off[g];
  const int64_t loff = p.pp.lap_off[g];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  SweepCtx c;
  c.alpha = p.alpha[0];
  c.paper = p.paper != 0;
  c.reslap = p.reslap != 0;
  c.has_prev = c.reslap && p.Lprev != nullptr;
  c.beta = c.has_prev ? p.beta[0] : 0.f;
  c.s1 = 1.f; c.s2 = 1.f; c.k2 = 0.f;
  if (PASS != SW_NORM) {
    c.s1 = p.stats[4 * g + 0];
    c.s2 = p.stats[4 * g + 1];
  }
  if (PASS == SW_B2) c.k2 = p.gstat[4 * g + 0];
  c.clipped2 = c.s2 < 1.f;
  const bool rd_dist = c.paper;
  const bool rd_lint = PASS == SW_NORM ? c.reslap : (PASS == SW_B2 ? (c.reslap && c.clipped2) : true);
  const bool rd_prev = c.has_prev;
  const bool rd_dl = PASS == SW_B1 || PASS == SW_B2;
  float part[4] = {0.f, 0.f, 0.f, 0.f};
  // rows of 4-float quads when the graph's rows are 16-byte aligned (every equal-size cloud); scalars otherwise
  const bool vec = (n & 3) == 0 && (loff & 3) == 0 && (row0 & 3) == 0;
  for (int r = 0; r < 8; ++r) {
    const int i = m0 + wid * 8 + r;
    if (i >= n) break;
    const float dis_i = c.paper ? p.dis[row0 + i] : 0.f;
    const int64_t base = loff + (int64_t)i * n;
    if (vec) {
#pragma unroll 2
      for (int j = 4 * lane; j < n; j += 128) {
        const int64_t idx = base + j;
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 dist = rd_dist ? ldg4(p.dist + idx) : z4;
        const float4 lint = rd_lint ? ldg4(p.Lint + idx) : z4;
        const float4 prev = rd_prev ? ldg4(p.Lprev + idx) : z4;
        const float4 gd = rd_dl ? *reinterpret_cast<const float4*>(p.dL + idx) : z4;
        const float4 dj = c.paper ? ldg4(p.dis + row0 + j) : z4;
        float4 resl, lall, dl, dlp;
        sweep_elem<PASS>(c, i == j, dis_i, dj.x, dist.x, lint.x, prev.x, gd.x, part, resl.x, lall.x, dl.x, dlp.x);
        sweep_elem<PASS>(c, i == j + 1, dis_i, dj.y, dist.y, lint.y, prev.y, gd.y, part, resl.y, lall.y, dl.y, dlp.y);
        sweep_elem<PASS>(c, i == j + 2, dis_i, dj.z, dist.z, lint.z, prev.z, gd.z, part, resl.z, lall.z, dl.z, dlp.z);
        sweep_elem<PASS>(c, i == j + 3, dis_i, dj.w, dist.w, lint.w, prev.w, gd.w, part, resl.w, lall.w, dl.w, dlp.w);
        if (PASS == SW_FINAL) {
          if (p.resL) stg4(p.resL + idx, resl);
          if (p.Lall) stg4(p.Lall + idx, lall);
          if (p.Lall2) stg4(p.Lall2 + idx, lall);
        } else if (PASS != SW_NORM) {
          stg4(p.dL + idx, dl);
          if (PASS == SW_B2 && c.has_prev && p.dLprev) stg4(p.dLprev + idx, dlp);
        }
      }
    } else {
#pragma unroll 4
      for (int j = lane; j < n; j += 32) {
        const int64_t idx = base + j;
        const float dist = rd_dist ? p.dist[idx] : 0.f;
        const float lint = rd_lint ? p.Lint[idx] : 0.f;
        const float prev = rd_prev ? p.Lprev[idx] : 0.f;
        const float gd = rd_dl ? p.dL[idx] : 0.f;
        const float dj = c.paper ? p.dis[row0 + j] : 0.f;
        float resl, lall, dl, dlp;
        sweep_elem<PASS>(c, i == j, dis_i, dj, dist, lint, prev, gd, part, resl, lall, dl, dlp);
        if (PASS == SW_FINAL) {
          if (p.resL) p.resL[idx] = resl;
          if (p.Lall) p.Lall[idx] = lall;
          if (p.Lall2) p.Lall2[idx] = lall;
        } else if (PASS != SW_NORM) {
          p.dL[idx] = dl;
          if (PASS == SW_B2 && c.has_prev && p.dLprev) p.dLprev[idx] = dlp;
        }
      }
    }
  }
  if (PASS == SW_FINAL) return;
  block_sum_vec<4>(part, red);
  if (threadIdx.x == 0) {
    float* tp = p.tilepart + (int64_t)t * 8 + (PASS == SW_B2 ? 4 : 0);
    tp[0] = part[0]; tp[1] = part[1]; tp[2] = part[2]; tp[3] = part[3];
  }
}

// per big graph: fold the tile partials (fixed order) into the scalars the next sweep needs
enum { ST_FWD = 0, ST_B1 = 1, ST_B2 = 2 };

struct StatArgs {
  BigPtrs pp;
  int variant, reslap, has_prev;
  const float* tilepart;
  float* stats;
  float* gstat;
  float* dalpha_part;
  float* dbeta_part;
};

template <int WHICH>
__global__ void big_stats_kernel(StatArgs p) {
  const int bi = blockIdx.x;
  const int g = p.pp.order[bi];
  const int n = p.pp.n_nodes[g];
  const int t0 = p.pp.big_tile_start[bi], t1 = p.pp.big_tile_start[bi + 1];
  const int lane = threadIdx.x;
  double s[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    double v = 0.0;
    for (int t = t0 + lane; t < t1; t += 32) v += (double)p.tilepart[(int64_t)t * 8 + k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    s[k] = v;
  }
  if (lane != 0) return;
  if (WHICH == ST_FWD) {
    // tf.clip_by_average_norm (graphconv.py:212) / tf.clip_by_norm (graphconv_reslap.py:185)
    const float normR2 = (float)s[0];
    const float inv1 = (normR2 > 0.f) ? rsqrtf(normR2) : INFINITY;
    const float s1 = (p.variant == AGCN_VARIANT_SGC_LL) ? fminf(inv1 * (float)n * (float)n, 1.f) : fminf(inv1, 1.f);
    float s2 = 1.f, normZ2 = 0.f;
    if (p.reslap) {
      // Z = s1 leaky(R) + C  (leaky(s R) = s leaky(R) for s > 0):  |Z|^2 from the three quadratic forms
      normZ2 = (float)((double)s1 * s1 * s[1] + 2.0 * s1 * s[2] + s[3]);
      const float inv2 = (normZ2 > 0.f) ? rsqrtf(normZ2) : INFINITY;
      s2 = fminf(inv2, 1.f);  // graphconv_reslap.py:194
    }
    p.stats[4 * g + 0] = s1;
    p.stats[4 * g + 1] = s2;
    p.stats[4 * g + 2] = normR2;
    p.stats[4 * g + 3] = normZ2;
  } else if (WHICH == ST_B1) {
    const float s2 = p.stats[4 * g + 1];
    p.gstat[4 * g + 0] = (s2 < 1.f) ? s2 * s2 * s2 * (float)s[1] : 0.f;  // k2
  } else {
    const float s1 = p.stats[4 * g + 0];
    const float cavg = (p.variant == AGCN_VARIANT_SGC_LL) ? (float)n * (float)n : 1.f;
    p.gstat[4 * g + 1] = (s1 < 1.f) ? (s1 * s1 * s1 / (cavg * cavg)) * (float)s[6] : 0.f;  // k1
    p.dalpha_part[g] = (float)((p.reslap ? s[0] : 0.0) + s[4]);
    if (p.dbeta_part) p.dbeta_part[g] = p.has_prev ? (float)s[5] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------
// metric block backward (paper semantics, metric_grad = full): sweeps that need element (i,j) and (j,i)
// ------------------------------------------------------------------------------------------------
// Everything here is symmetric in (i, j) up to the pair (gu_ij, gu_ji): W, dist and R are, and so are the summands
//   e_ij = (dR_ij + dR_ji) W_ij                      -> d dis_m = -sum_j e_mj dis_j                       (TR_DD)
//   C_ij = -W_ij (dW_ij + dW_ji) / dist_ij = C_ji                                                        (TR_C)
// so one CTA takes a PAIR of 64 x 64 tiles (I, J), I <= J: it reads gu[I, J], gu[J, I] and dist[I, J] once, writes C[I, J]
// and (transposed through shared memory) C[J, I], and leaves the sums over its columns for the rows of I and over its
// rows for the rows of J as partials part[row][column block] -- each (row, block) is written by exactly one CTA, a
// second kernel adds them in block order (deterministic, no atomics).
enum { TR_DD = 0, TR_C = 1 };

struct TransArgs {
  BigPtrs pp;
  const float* dist;
  const float* dis;
  const float* stats;
  const float* gstat;
  const float* gu;  // d(s1 R) after the leaky rectifier (in the dL scratch)
  float* dd;        // [R] gradient w.r.t. the degree d_m
  float* C;         // packed: C_ij = (d dist_ij + d dist_ji) / dist_ij
  float* rs;        // [R] rowsum(C)
  float* part;      // [R][ncb]
  int ncb;
};

template <int PASS>
__global__ void __launch_bounds__(256, PASS == TR_C ? 4 : 5) big_trans_kernel(TransArgs p) {
  __shared__ float sA[PT][PT + 1];   // gu[I, J]
  __shared__ float sB[PT][PT + 1];   // gu[J, I]; then C[J, I]
  __shared__ float scol[8][PT];
  const int t = blockIdx.x;
  const int g = p.pp.tile_graph[t], m0 = p.pp.tile_row[t];
  const int n = p.pp.n_nodes[g];
  const int j0 = blockIdx.y * PT;
  if (j0 < m0 || j0 >= n) return;
  const bool diag_tile = j0 == m0;
  const int64_t row0 = p.pp.node_off[g];
  const int64_t loff = p.pp.lap_off[g];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const float s1 = p.stats[4 * g + 0];
  const float k1 = p.gstat[4 * g + 1];
  const bool clipped1 = s1 < 1.f;
  if ((n & 3) == 0 && (loff & 3) == 0) {
    for (int e = threadIdx.x; e < PT * PT / 4; e += 256) {
      const int a = e / (PT / 4), b = 4 * (e % (PT / 4));
      const int i = m0 + a, j = j0 + b;   // rows of n % 4 == 0 floats: a quad is inside or outside as a whole
      const float4 va = (i < n && j < n) ? __ldg(reinterpret_cast<const float4*>(p.gu + loff + (int64_t)i * n + j))
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
      sA[a][b] = va.x; sA[a][b + 1] = va.y; sA[a][b + 2] = va.z; sA[a][b + 3] = va.w;
      const int jj = j0 + a, ii = m0 + b;
      const float4 vb = (jj < n && ii < n) ? __ldg(reinterpret_cast<const float4*>(p.gu + loff + (int64_t)jj * n + ii))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
      sB[a][b] = vb.x; sB[a][b + 1] = vb.y; sB[a][b + 2] = vb.z; sB[a][b + 3] = vb.w;
    }
  } else {
    for (int e = threadIdx.x; e < PT * PT; e += 256) {
      const int a = e / PT, b = e % PT;
      const int i = m0 + a, j = j0 + b;
      sA[a][b] = (i < n && j < n) ? p.gu[loff + (int64_t)i * n + j] : 0.f;
      const int jj = j0 + a, ii = m0 + b;
      sB[a][b] = (jj < n && ii < n) ? p.gu[loff + (int64_t)jj * n + ii] : 0.f;
    }
  }
  __syncthreads();
  float colacc[2] = {0.f, 0.f};
  float dis_j[2], dd_j[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int j = j0 + lane + 32 * h;
    dis_j[h] = j < n ? p.dis[row0 + j] : 0.f;
    dd_j[h] = (PASS == TR_C && j < n) ? p.dd[row0 + j] : 0.f;
  }
  float dst[8][2];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = m0 + wid * 8 + r, j = j0 + lane + 32 * h;
      dst[r][h] = (i < n && j < n) ? __ldg(p.dist + loff + (int64_t)i * n + j) : 0.f;
    }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int a = wid * 8 + r, i = m0 + a;
    const bool row_ok = i < n;
    const float dis_i = row_ok ? p.dis[row0 + i] : 0.f;
    const float dd_i = (PASS == TR_C && row_ok) ? p.dd[row0 + i] : 0.f;
    float rowacc = 0.f;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int b = lane + 32 * h, j = j0 + b;
      float val = 0.f;   // e_ij | C_ij
      if (row_ok && j < n && j != i) {
        const float w = expf(-dst[r][h]);
        const float R = -(dis_i * w) * dis_j[h];
        float g_ij = sA[a][b], g_ji = sB[b][a];
        if (clipped1) {  // s1 = c |R|^-1: dR = s1 gu - R (s1^3 / c^2) <gu, R>
          g_ij = s1 * g_ij - R * k1;
          g_ji = s1 * g_ji - R * k1;
        }
        if (PASS == TR_DD) {
          // d dis_m = -sum_j dR_mj W_mj dis_j - sum_j dR_jm W_jm dis_j
          val = (g_ij + g_ji) * w;
          rowacc += val * dis_j[h];
          colacc[h] += val * dis_i;
        } else {
          const float dw_ij = -g_ij * dis_i * dis_j[h] + dd_j[h];
          const float dw_ji = -g_ji * dis_i * dis_j[h] + dd_i;
          const float ddist = -w * (dw_ij + dw_ji);
          val = (dst[r][h] > 0.f) ? ddist / dst[r][h] : 0.f;  // sub-gradient 0 at exact duplicates (SURVEY H5)
          rowacc += val;
          colacc[h] += val;
        }
      }
      if (PASS == TR_C) {
        if (row_ok && j < n) p.C[loff + (int64_t)i * n + j] = val;   // the diagonal gets its 0 here
        sB[b][a] = val;   // same thread read this element: no hazard
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rowacc += __shfl_xor_sync(0xffffffffu, rowacc, o);
    if (lane == 0 && row_ok) p.part[(row0 + i) * p.ncb + blockIdx.y] = rowacc;
  }
  if (diag_tile) return;   // the row sums covered every pair of this tile
  scol[wid][lane] = colacc[0];
  scol[wid][lane + 32] = colacc[1];
  __syncthreads();
  if (threadIdx.x < PT) {
    const int j = j0 + threadIdx.x;
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) v += scol[k][threadIdx.x];
    if (j < n) p.part[(row0 + j) * p.ncb + m0 / PT] = v;
  }
  if (PASS == TR_C) {
    for (int e = threadIdx.x; e < PT * PT; e += 256) {
      const int b = e / PT, a = e % PT;   // row j0 + b of C, columns m0 + a
      if (j0 + b < n && m0 + a < n) p.C[loff + (int64_t)(j0 + b) * n + m0 + a] = sB[b][a];
    }
  }
}

// fold the column-block partials of a row (block order) into dd (TR_DD) or rowsum(C) (TR_C)
template <int PASS>
__global__ void big_trans_fold_kernel(TransArgs p) {
  const int t = blockIdx.x;
  const int g = p.pp.tile_graph[t], i = p.pp.tile_row[t] + threadIdx.x;
  const int n = p.pp.n_nodes[g];
  if (i >= n) return;
  const int64_t row = p.pp.node_off[g] + i;
  const int nb = (n + PT - 1) / PT;
  float v = 0.f;
  for (int b = 0; b < nb; ++b) v += p.part[row * p.ncb + b];
  if (PASS == TR_DD) {
    const float dm = p.dis[row];
    p.dd[row] = -0.5f * dm * dm * dm * (-v);  // dd_m = -1/2 dis_m^3 d dis_m  (0 when d_m == 0)
  } else {
    p.rs[row] = v;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
namespace {
struct BigWork {
  float *rowpart, *tilepart, *gstat, *stats_tmp, *norms, *dd, *rs, *C;
  int ncb;
  size_t bytes;
};
BigWork carve_big(const agcn_plan* plan, float* base, bool full) {
  Arena c(base);
  BigWork w{};
  w.ncb = (plan->max_n + PT - 1) / PT;
  w.rowpart = c.take((size_t)plan->R * w.ncb);
  w.tilepart = c.take((size_t)plan->big_tiles * 8);
  w.gstat = c.take((size_t)plan->B * 4);
  w.stats_tmp = c.take((size_t)plan->B * 4);
  w.norms = c.take((size_t)plan->R);
  c.take((size_t)plan->B * 256);  // per-graph mean rows behind the norms (tensor-core pair kernel, F <= 256)
  if (full) {
    w.dd = c.take((size_t)plan->R);
    w.rs = c.take((size_t)plan->R);
    w.C = c.take((size_t)plan->LL);
  }
  w.bytes = c.bytes;
  return w;
}
}  // namespace

size_t big_work_floats(const agcn_plan* plan, bool full) {
  if (plan->large_count == 0) return 0;
  return carve_big(plan, nullptr, full).bytes / sizeof(float);
}

int big_build_laplacian(const GraphArgs& a, bool need_W, float* big_work, cudaStream_t st) {
  const agcn_plan* plan = a.plan;
  if (plan->large_count == 0) return AGCN_OK;
  const bool paper = a.lap_mode == AGCN_LAP_PAPER;
  const bool reslap = a.variant == AGCN_VARIANT_SGC_LL_RESLAP;
  BigWork w = carve_big(plan, big_work, false);
  const BigPtrs pp = big_ptrs(plan);
  const int tiles = plan->big_tiles;
  if (need_W) {
    if (pair_tc_supported(plan, a.F)) {
      // equal-size clouds: Gram tiles on the tensor cores, direct-difference fix-up for near-duplicates (agcn_big_tc.cu)
      int rc = pair_tc_similarity(plan, a.XW, a.F, w.norms, a.dist, a.resW, paper ? w.rowpart : nullptr, w.ncb, st);
      if (rc) return rc;
    } else {
      PairArgs k{};
      k.pp = pp; k.F = a.F; k.XW = a.XW; k.dist = a.dist; k.resW = a.resW;
      k.rowpart = paper ? w.rowpart : nullptr; k.ncb = w.ncb;
      dim3 grid(tiles, w.ncb);
      {
        ProfScope prof("big_pair_kernel<SIM>", st);
        big_pair_kernel<PAIR_SIM><<<grid, 256, 0, st>>>(k);
      }
      AGCN_LAUNCH_CHECK();
    }
    if (paper) {
      big_dis_kernel<<<tiles, PT, 0, st>>>(pp, w.rowpart, w.ncb, a.dis);
      AGCN_LAUNCH_CHECK();
    }
  }
  // literal SGC_LL keeps no statistics for backward (L_all = I + L_int); its optional outputs still need them
  float* stats = a.stats ? a.stats : w.stats_tmp;
  if (!a.stats && !a.resL && !a.Lall && !a.Lall_out) return AGCN_OK;
  SweepArgs s{};
  s.pp = pp; s.paper = paper ? 1 : 0; s.reslap = reslap ? 1 : 0;
  s.dist = a.dist; s.dis = a.dis; s.Lint = a.Lint; s.Lprev = reslap ? a.Lprev : nullptr;
  s.alpha = a.alpha; s.beta = a.beta; s.stats = stats;
  s.resL = a.resL; s.Lall = a.Lall; s.Lall2 = a.Lall_out; s.tilepart = w.tilepart;
  {
    ProfScope prof("big_sweep_kernel", st);
    big_sweep_kernel<SW_NORM><<<tiles, 256, 0, st>>>(s);
  }
  AGCN_LAUNCH_CHECK();
  StatArgs q{};
  q.pp = pp; q.variant = a.variant; q.reslap = reslap ? 1 : 0; q.has_prev = (reslap && a.Lprev) ? 1 : 0;
  q.tilepart = w.tilepart; q.stats = stats; q.gstat = w.gstat;
  big_stats_kernel<ST_FWD><<<plan->large_count, 32, 0, st>>>(q);
  AGCN_LAUNCH_CHECK();
  {
    ProfScope prof("big_sweep_kernel", st);
    big_sweep_kernel<SW_FINAL><<<tiles, 256, 0, st>>>(s);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// dL = dLall_in + sum_{k=1}^{K-1} c_k U_k T_{k-1}^T for the big graphs; U_k = slice k of G (after the
// in-place reverse recurrence)
int big_dL(const GraphArgs& a, const float* U, cudaStream_t st) {
  const agcn_plan* plan = a.plan;
  if (plan->large_count == 0) return AGCN_OK;
  if (a.K >= 2 && pair_tc_supported(plan, a.F) && ((reinterpret_cast<uintptr_t>(a.dL) | reinterpret_cast<uintptr_t>(a.dLall_in)) & 15) == 0)
    return pair_tc_dL(plan, U, a.X, a.T, a.F, a.K, a.dLall_in, a.dL, st);
  PairArgs k{};
  k.pp = big_ptrs(plan); k.F = a.F;
  k.S = a.K - 1; k.U = U; k.X = a.X; k.T = a.T; k.slice = (int64_t)plan->R * a.F;
  k.dL_in = a.dLall_in; k.dL = a.dL;
  dim3 grid(plan->big_tiles, (plan->max_n + PT - 1) / PT);
  {
    ProfScope prof("big_pair_kernel<DL>", st);
    big_pair_kernel<PAIR_DL><<<grid, 256, 0, st>>>(k);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

int grouped_rows_gemm(const agcn_plan* plan, int tiles, const float* Lmat, const float* In, float cmul,
                      const float* row_scale, const float* scale_in, float* Out, int F, cudaStream_t st);

int big_laplacian_bwd(const GraphArgs& a, float* big_work, cudaStream_t st) {
  const agcn_plan* plan = a.plan;
  if (plan->large_count == 0) return AGCN_OK;
  const bool paper = a.lap_mode == AGCN_LAP_PAPER;
  const bool reslap = a.variant == AGCN_VARIANT_SGC_LL_RESLAP;
  const bool full = paper && a.metric_full;
  BigWork w = carve_big(plan, big_work, full);
  const BigPtrs pp = big_ptrs(plan);
  const int tiles = plan->big_tiles;
  SweepArgs s{};
  s.pp = pp; s.paper = paper ? 1 : 0; s.reslap = reslap ? 1 : 0;
  s.dist = a.dist; s.dis = a.dis; s.Lint = a.Lint; s.Lprev = reslap ? a.Lprev : nullptr;
  s.alpha = a.alpha; s.beta = a.beta; s.stats = a.stats; s.gstat = w.gstat;
  s.dL = a.dL; s.dLprev = a.dLprev; s.tilepart = w.tilepart;
  StatArgs q{};
  q.pp = pp; q.variant = a.variant; q.reslap = reslap ? 1 : 0; q.has_prev = (reslap && a.Lprev) ? 1 : 0;
  q.tilepart = w.tilepart; q.stats = a.stats; q.gstat = w.gstat;
  q.dalpha_part = a.dalpha_part; q.dbeta_part = a.dbeta_part;
  if (reslap) {
    {
      ProfScope prof("big_sweep_kernel", st);
      big_sweep_kernel<SW_B1><<<tiles, 256, 0, st>>>(s);
    }
    AGCN_LAUNCH_CHECK();
    big_stats_kernel<ST_B1><<<plan->large_count, 32, 0, st>>>(q);
    AGCN_LAUNCH_CHECK();
  }
  {
    ProfScope prof("big_sweep_kernel", st);
    big_sweep_kernel<SW_B2><<<tiles, 256, 0, st>>>(s);
  }
  AGCN_LAUNCH_CHECK();
  big_stats_kernel<ST_B2><<<plan->large_count, 32, 0, st>>>(q);
  AGCN_LAUNCH_CHECK();
  if (!full) return AGCN_OK;
  TransArgs t{};
  t.pp = pp; t.dist = a.dist; t.dis = a.dis; t.stats = a.stats; t.gstat = w.gstat; t.gu = a.dL;
  t.dd = w.dd; t.C = w.C; t.rs = w.rs; t.part = w.rowpart; t.ncb = w.ncb;   // rowpart: free in backward
  const dim3 pairs(tiles, w.ncb);
  {
    ProfScope prof("big_trans_kernel", st);
    big_trans_kernel<TR_DD><<<pairs, 256, 0, st>>>(t);
  }
  AGCN_LAUNCH_CHECK();
  big_trans_fold_kernel<TR_DD><<<tiles, PT, 0, st>>>(t);
  AGCN_LAUNCH_CHECK();
  {
    ProfScope prof("big_trans_kernel", st);
    big_trans_kernel<TR_C><<<pairs, 256, 0, st>>>(t);
  }
  AGCN_LAUNCH_CHECK();
  big_trans_fold_kernel<TR_C><<<tiles, PT, 0, st>>>(t);
  AGCN_LAUNCH_CHECK();
  // dXW_i = rowsum(C)_i xw_i - (C XW)_i
  return grouped_rows_gemm(plan, tiles, w.C, a.XW, -1.f, w.rs, a.XW, a.dXW, a.F, st);
}

}  // namespace agcn
