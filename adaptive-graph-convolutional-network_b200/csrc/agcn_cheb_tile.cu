// Chebyshev recurrences of the graphs up to AGCN_SMALL_MAX nodes as small, high-occupancy CUDA-core CTAs, split from the
// tensor-core transform (agcn_pre_tile.cu):
//
//   forward   T_0 = X, T_1 = L T_0, T_k = 2 L T_{k-1} - T_{k-2}            graphconv.py:221-236
//   backward  U_{K-1} = G_{K-1}, U_j = G_j + c_{j+1} L^T U_{j+1} - U_{j+2},  dX = U_0   (reverse mode of the same lines)
//
// Why split (profiles/r02f_*): the fused tile kernels of round 1 ran ONE 320-thread CTA per SM (222 KB of shared
// memory) through a serial chain of ~25 dependent phases per tile -- 26 us of worker chain against 6 us of tensor-core
// work per tile, 5 % of the HBM roofline -- and nothing else can be resident beside them to hide the latencies.  Here a
// CTA owns (tile, 32-column chunk): 256 threads (tile row x column half), ~74 KB of shared memory, three CTAs per SM, a
// grid four times the tile count, so every SM interleaves 24 warps of independent chains.  The transform then runs as a
// plain contraction over all packed rows at the tensor core's own pace (pt::pre_tile_kernel).
//
// Sparse rows: the Laplacian of a molecule has ~3 non-zeros per row (reference_literal mode multiplies by I + L_int, the
// normalised Laplacian of a graph of degree <= 4), so a dense n x n product spends 80 .. 95 % of its loads and FMAs on
// exact zeros.  Every thread keeps the non-zero pattern of its row (forward) / column (backward) as a bit mask and walks
// the set bits; the values stay in the dense shared-memory copy.  Skipping a term whose coefficient is exactly 0 does not
// change an fp32 sum of finite values.  Dense matrices (paper mode) take the dense loop, chosen per warp.
//
// Tiles: the plan's fused tiles (whole graphs with n <= AGCN_FUSE_MAX_N packed into 128 rows) or, for the graphs between
// AGCN_FUSE_MAX_N and AGCN_SMALL_MAX nodes, one graph per CTA row range (160 rows, 320 threads).
#include <algorithm>
#include <mutex>

#include "agcn_internal.cuh"

namespace agcn {
namespace ct {

constexpr int CH = 32;        // feature columns per CTA
constexpr int CPITCH = 144;   // bytes per row of a chunk buffer: 32 floats + 4 of padding

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];\n" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};\n" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t a, float v) {
  asm volatile("st.shared.f32 [%0], %1;\n" ::"r"(a), "f"(v) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t sdst, const float* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sdst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t sdst, const float* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sdst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

struct CtArgs {
  // graph list of a CTA: a fused tile of the plan (tile_graphs != NULL) or graph order[order_start + tile]
  const int4* tile_graphs;     // 2 x int4 per entry: {g, r0, n, lbase}, {node_off, lap_off lo, hi, 0}
  const int32_t* tile_gstart;
  const int32_t* order;
  const int32_t* n_nodes;
  const int32_t* node_off;
  const int64_t* lap_off;
  int order_start;
  int chunks;                  // 32-column chunks of F
  int cpc;                     // chunks per CTA, processed one after the other with the tile's L matrices and masks kept
  int groups;                  // ceil(chunks / cpc); grid = tiles * groups
  int rows;                    // row capacity of a CTA; blockDim.x == 2 * rows
  int lfloats;                 // floats of the shared-memory L region
  const float* L;              // packed Laplacians (Lint or L_all)
  int add_identity;
  int transL;                  // forward kernel: multiply by L^T (the V_k = T_k(L^T) dYpre recurrences of the backward pass)
  int F, K;
  const float* X;              // forward  [R, F]
  float* T;                    //          [K-1][R][F]
  long long tslice;
  const float* G;              // backward [K][R][F]  G_z = dYpre W_z^T
  long long gslice;
  float* dX;                   //          [R, F]
};

struct Row {
  int grow;   // packed row or -1
  int n;      // nodes of my graph (0: padding row)
  int r0;     // CTA row of my graph's first node
  int lbase;  // float offset of my graph's matrix in the L region
  int i;      // my index inside the graph
  int pitch;  // row pitch of the matrix (n | 1)
};

// n x n matrix (row-major, contiguous in global memory) -> shared memory with row pitch `pitch`: one warp per row, lanes
// along the row, left in flight (cp.async; a register-staged LDG + STS copy measured slower: 37 against 31 us per launch)
__device__ __forceinline__ void copy_matrix(const float* __restrict__ src, uint32_t dst, int n, int pitch) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int i = warp; i < n; i += nw) {
    const float* srow = src + (long long)i * n;
    const uint32_t drow = dst + 4 * (i * pitch);
    for (int j = lane; j < n; j += 32) cp_async4(drow + 4 * j, srow + j);
  }
}

// Graph list + row table of the CTA; the L matrices are complete after the next __syncthreads.
template <bool TILE>
__device__ __forceinline__ Row prologue(const CtArgs& p, int tile, int r, uint32_t s_glist, uint32_t sL) {
  Row t;
  t.grow = -1; t.n = 0; t.r0 = 0; t.lbase = 0; t.i = 0; t.pitch = 1;
  const int tid = threadIdx.x, nthreads = blockDim.x;
  if (TILE) {
    // ONE warp fetches the tile's graph list: with every thread of 444 resident CTAs reading the same few cache lines of
    // the plan tables, the first phase of the kernel took 5 us (per-CTA globaltimer timeline)
    if (tid < 32) {
      int gs = 0, ge = 0;
      if (tid == 0) {
        gs = __ldg(p.tile_gstart + tile);
        ge = __ldg(p.tile_gstart + tile + 1);
      }
      gs = __shfl_sync(0xffffffffu, gs, 0);
      ge = __shfl_sync(0xffffffffu, ge, 0);
      const int ng2 = 2 * (ge - gs);
      for (int e = tid; e < ng2; e += 32) {
        const int4 v = __ldg(p.tile_graphs + 2 * gs + e);
        asm volatile("st.shared.v4.s32 [%0], {%1,%2,%3,%4};\n" ::"r"(s_glist + 16 * e), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
      }
      if (tid == 0) asm volatile("st.shared.s32 [%0], %1;\n" ::"r"(s_glist + 128 * 32), "r"(ge - gs) : "memory");
    }
    __syncthreads();
    int ng;
    asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(ng) : "r"(s_glist + 128 * 32) : "memory");
    for (int e = 0; e < ng; ++e) {
      int gx, gy, gz, gw, noff, lo, hi, pad;
      asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];\n" : "=r"(gx), "=r"(gy), "=r"(gz), "=r"(gw) : "r"(s_glist + 32 * e) : "memory");
      asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];\n" : "=r"(noff), "=r"(lo), "=r"(hi), "=r"(pad) : "r"(s_glist + 32 * e + 16) : "memory");
      if (r >= gy && r < gy + gz) {
        t.grow = noff + (r - gy);
        t.n = gz; t.r0 = gy; t.lbase = gw; t.i = r - gy; t.pitch = gz | 1;
      }
      // this graph's matrix, row pitch n | 1 (odd: rows read by neighbouring lanes sit in different banks): one warp per
      // row, lanes along the row (coalesced, two or three instructions per element instead of an index walk)
      const long long loff = (long long)(((unsigned long long)(unsigned)hi << 32) | (unsigned)lo);
      copy_matrix(p.L + loff, sL + 4 * gw, gz, gz | 1);
    }
  } else {
    const int g = p.order[p.order_start + tile];
    const int n = p.n_nodes[g], pitch = n | 1;
    if (r < n) {
      t.grow = p.node_off[g] + r;
      t.n = n; t.i = r; t.pitch = pitch;
    }
    copy_matrix(p.L + p.lap_off[g], sL, n, pitch);
  }
  cp_async_commit();
  return t;
}

// non-zero pattern of a row / column: MW 32-bit words
template <int MW>
struct Mask {
  uint32_t w[MW];
};

template <int MW>
__device__ __forceinline__ Mask<MW> nonzero_mask(uint32_t laddr, int lstride_bytes, int n) {
  Mask<MW> m;
#pragma unroll
  for (int k = 0; k < MW; ++k) {
    uint32_t bits = 0;
    const int j0 = 32 * k;
    if (j0 < n) {
      const int cnt = min(32, n - j0);
      uint32_t a = laddr + (uint32_t)(j0 * lstride_bytes);
      int j = 0;
      for (; j + 8 <= cnt; j += 8) {   // eight loads in flight, constant bit positions
        uint32_t b8 = 0;
#pragma unroll
        for (int u = 0; u < 8; ++u) b8 |= (lds32(a + (uint32_t)(u * lstride_bytes)) != 0.f) ? (1u << u) : 0u;
        bits |= b8 << j;
        a += 8 * lstride_bytes;
      }
      for (; j < cnt; ++j) {
        bits |= (lds32(a) != 0.f) ? (1u << j) : 0u;
        a += lstride_bytes;
      }
    }
    m.w[k] = bits;
  }
  return m;
}
// Warp-uniform choice between the dense loop (n x ~21 instructions) and the masked loop (~28 per non-zero)
template <int MW>
__device__ __forceinline__ bool prefer_masked(const Mask<MW>& m, int n) {
  int nnz = 0;
#pragma unroll
  for (int k = 0; k < MW; ++k) nnz += __popc(m.w[k]);
  const unsigned dense_cost = __reduce_max_sync(0xffffffffu, (unsigned)(n * 3));
  const unsigned masked_cost = __reduce_max_sync(0xffffffffu, (unsigned)(nnz * 4));
  return masked_cost < dense_cost;
}

__device__ __forceinline__ void fma_row(float a, const float4 b[4], float acc[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    acc[4 * g] = fmaf(a, b[g].x, acc[4 * g]);
    acc[4 * g + 1] = fmaf(a, b[g].y, acc[4 * g + 1]);
    acc[4 * g + 2] = fmaf(a, b[g].z, acc[4 * g + 2]);
    acc[4 * g + 3] = fmaf(a, b[g].w, acc[4 * g + 3]);
  }
}
// acc[:] += sum_j L[laddr + j * lstride_bytes] * src[r0 + j][16h .. 16h+15]     (all j < n)
__device__ __forceinline__ void lap_times_rows(uint32_t laddr, int lstride_bytes, uint32_t src, int r0, int n, int h,
                                               float acc[16]) {
  uint32_t ta = src + (uint32_t)(r0 * CPITCH + h * 64);
  uint32_t la = laddr;
  int j = 0;
  for (; j < n; ++j) {
    const float a = lds32(la);
    float4 b[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) b[g] = lds128(ta + 16 * g);
    fma_row(a, b, acc);
    la += lstride_bytes;
    ta += CPITCH;
  }
}
// the same sum over the set bits of the mask only
template <int MW>
__device__ __forceinline__ void lap_times_rows_masked(uint32_t laddr, int lstride_bytes, uint32_t src, int r0,
                                                      const Mask<MW>& m, int h, float acc[16]) {
#pragma unroll
  for (int k = 0; k < MW; ++k) {
    uint32_t bits = m.w[k];
    const uint32_t tbase = src + (uint32_t)((r0 + 32 * k) * CPITCH + h * 64);
    const uint32_t lbase = laddr + (uint32_t)(32 * k * lstride_bytes);
    while (bits) {   // one term per trip: the other resident warps (24 per SM) cover the shared-memory latency
      const int j = __ffs((int)bits) - 1;
      bits &= bits - 1;
      const float a = lds32(lbase + (uint32_t)(j * lstride_bytes));
      float4 b[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) b[g] = lds128(tbase + (uint32_t)(j * CPITCH + 16 * g));
      fma_row(a, b, acc);
    }
  }
}

__device__ __forceinline__ uint32_t seg_addr(uint32_t buf, int row, int h) { return buf + (uint32_t)(row * CPITCH + h * 64); }
__device__ __forceinline__ void read_seg(uint32_t buf, int row, int h, float v[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float4 x = lds128(seg_addr(buf, row, h) + 16 * g);
    v[4 * g] = x.x; v[4 * g + 1] = x.y; v[4 * g + 2] = x.z; v[4 * g + 3] = x.w;
  }
}
__device__ __forceinline__ void write_seg(uint32_t buf, int row, int h, const float v[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g)
    sts128(seg_addr(buf, row, h) + 16 * g, make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]));
}
// my 16 columns of a packed row, registers <-> global
__device__ __forceinline__ void load_seg(const float* __restrict__ M, int F, int grow, int col0, bool vec, float v[16]) {
  if (grow < 0) {
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = 0.f;
    return;
  }
  const float* src = M + (long long)grow * F + col0;
  if (vec) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col0 + 4 * g < F) x = __ldg(reinterpret_cast<const float4*>(src) + g);
      v[4 * g] = x.x; v[4 * g + 1] = x.y; v[4 * g + 2] = x.z; v[4 * g + 3] = x.w;
    }
  } else {
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = (col0 + u < F) ? __ldg(src + u) : 0.f;
  }
}
__device__ __forceinline__ void store_seg(float* __restrict__ M, int F, int grow, int col0, bool vec, const float v[16]) {
  if (grow < 0) return;
  float* dst = M + (long long)grow * F + col0;
  if (vec) {
#pragma unroll
    for (int g = 0; g < 4; ++g)
      if (col0 + 4 * g < F)
        reinterpret_cast<float4*>(dst)[g] = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
  } else {
#pragma unroll
    for (int u = 0; u < 16; ++u)
      if (col0 + u < F) dst[u] = v[u];
  }
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
template <bool TILE, int MW>
__global__ void __launch_bounds__(TILE ? 256 : 320, TILE ? 3 : 1) cheb_tile_fwd_kernel(CtArgs p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int rows = p.rows;
  const uint32_t buf0 = sbase, buf1 = sbase + (uint32_t)(rows * CPITCH), sL = buf1 + (uint32_t)(rows * CPITCH),
                 s_glist = sL + 4u * (uint32_t)p.lfloats;
  const int tile = blockIdx.x / p.groups, grp = blockIdx.x - tile * p.groups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpr = rows >> 5;
  const int h = warp / wpr, r = (warp - h * wpr) * 32 + lane;
  const int F = p.F, K = p.K;
  const Row me = prologue<TILE>(p, tile, r, s_glist, sL);
  const bool vec = ((F & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.X) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(p.T) & 15) == 0) && ((p.tslice & 3) == 0);
  // my row of the graph's matrix, or (transL) my column: (L^T V)_i = sum_j L[j][i] V_j
  const uint32_t lrow = p.transL ? sL + 4 * (me.lbase + me.i) : sL + 4 * (me.lbase + me.i * me.pitch);
  const int lstep = p.transL ? 4 * me.pitch : 4;
  Mask<MW> mask;
  bool masked = false;
  const int c_beg = grp * p.cpc, c_end = min(p.chunks, c_beg + p.cpc);
  for (int c = c_beg; c < c_end; ++c) {
    const int col0 = c * CH + 16 * h;
    // T_0: my 16 columns -> my row segment of buf0
    {
      const uint32_t d = seg_addr(buf0, r, h);
      const float* src = p.X + (long long)(me.grow < 0 ? 0 : me.grow) * F + col0;
      if (vec) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (me.grow >= 0 && col0 + 4 * g < F)
            cp_async16(d + 16 * g, src + 4 * g);
          else
            sts128(d + 16 * g, make_float4(0.f, 0.f, 0.f, 0.f));
        }
      } else {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          if (me.grow >= 0 && col0 + u < F)
            cp_async4(d + 4 * u, src + u);
          else
            sts32(d + 4 * u, 0.f);
        }
      }
      cp_async_commit();
    }
    cp_async_wait_all();
    __syncthreads();  // (first chunk: the L matrices and) the T_0 chunk of every row have landed
    if (c == c_beg) {
      mask = nonzero_mask<MW>(lrow, lstep, me.n);
      masked = prefer_masked<MW>(mask, me.n);
    }
    float tm1[16], tm2[16];
    read_seg(buf0, r, h, tm1);
#pragma unroll
    for (int u = 0; u < 16; ++u) tm2[u] = 0.f;
    uint32_t src = buf0, dst = buf1;
    for (int s = 1; s < K; ++s) {
      float t[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) t[u] = p.add_identity ? tm1[u] : 0.f;  // L_all = I + L_int (literal mode)
      if (masked)
        lap_times_rows_masked<MW>(lrow, lstep, src, me.r0, mask, h, t);
      else
        lap_times_rows(lrow, lstep, src, me.r0, me.n, h, t);             // graphconv.py:231
      if (s >= 2) {
#pragma unroll
        for (int u = 0; u < 16; ++u) t[u] = 2.f * t[u] - tm2[u];          // graphconv.py:234
      }
      store_seg(p.T + (long long)(s - 1) * p.tslice, F, me.grow, col0, vec, t);
      if (s + 1 < K) {
        write_seg(dst, r, h, t);
        __syncthreads();  // T_s rows of every graph of the CTA are in `dst`; everybody is done reading `src`
        const uint32_t tmp = src; src = dst; dst = tmp;
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) { tm2[u] = tm1[u]; tm1[u] = t[u]; }
    }
    if (c + 1 < c_end) __syncthreads();  // the last step's reads are done before the next chunk lands in buf0
  }
}

// ------------------------------------------------------------------------------------------------
// backward (dX chain)
// ------------------------------------------------------------------------------------------------
template <bool TILE, int MW>
__global__ void __launch_bounds__(TILE ? 256 : 320, TILE ? 3 : 1) cheb_tile_bwd_kernel(CtArgs p) {
  extern __shared__ __align__(16) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int rows = p.rows;
  const uint32_t buf0 = sbase, buf1 = sbase + (uint32_t)(rows * CPITCH), sL = buf1 + (uint32_t)(rows * CPITCH),
                 s_glist = sL + 4u * (uint32_t)p.lfloats;
  const int tile = blockIdx.x / p.groups, grp = blockIdx.x - tile * p.groups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpr = rows >> 5;
  const int h = warp / wpr, r = (warp - h * wpr) * 32 + lane;
  const int F = p.F, K = p.K;
  const Row me = prologue<TILE>(p, tile, r, s_glist, sL);
  const bool vec = ((F & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.G) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(p.dX) & 15) == 0) && ((p.gslice & 3) == 0);
  cp_async_wait_all();
  __syncthreads();  // L matrices have landed
  const uint32_t lcol = sL + 4 * (me.lbase + me.i);  // column i of my graph's matrix: (L^T U)_i = sum_j L[j][i] U_j
  const Mask<MW> mask = nonzero_mask<MW>(lcol, 4 * me.pitch, me.n);
  const bool masked = prefer_masked<MW>(mask, me.n);
  const uint32_t ub[2] = {buf0, buf1};
  const int c_beg = grp * p.cpc, c_end = min(p.chunks, c_beg + p.cpc);
  for (int c = c_beg; c < c_end; ++c) {
    const int col0 = c * CH + 16 * h;
    float u1[16], u2[16];
    load_seg(p.G + (long long)(K - 1) * p.gslice, F, me.grow, col0, vec, u1);  // U_{K-1} = G_{K-1}
#pragma unroll
    for (int u = 0; u < 16; ++u) u2[u] = 0.f;
    int cur = 0;
    for (int j = K - 2; j >= 0; --j) {
      write_seg(ub[cur], r, h, u1);
      __syncthreads();  // U_{j+1} rows of every graph of the CTA are visible (two buffers: one barrier per step)
      float acc[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) acc[u] = p.add_identity ? u1[u] : 0.f;  // (I + L)^T U = U + L^T U
      if (masked)
        lap_times_rows_masked<MW>(lcol, 4 * me.pitch, ub[cur], me.r0, mask, h, acc);
      else
        lap_times_rows(lcol, 4 * me.pitch, ub[cur], me.r0, me.n, h, acc);
      const float cmul = (j + 1 >= 2) ? 2.f : 1.f;
#pragma unroll
      for (int u = 0; u < 16; ++u) acc[u] = cmul * acc[u] - u2[u];
      float g[16];   // loaded late: u1, u2, acc and the product's operands already fill the 80 registers of 3 CTAs / SM
      load_seg(p.G + (long long)j * p.gslice, F, me.grow, col0, vec, g);
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const float o = g[u] + acc[u];
        u2[u] = u1[u];
        u1[u] = o;
      }
      cur ^= 1;
    }
    store_seg(p.dX, F, me.grow, col0, vec, u1);  // dX = U_0
    if (c + 1 < c_end) __syncthreads();  // the last step's reads are done before the next chunk overwrites the buffers
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static size_t smem_bytes(int rows, int lfloats, bool tile) {
  return (size_t)2 * rows * CPITCH + (size_t)lfloats * 4 + (tile ? 128 * 32 + 16 : 0) + 64;
}

template <typename Kern>
static int opt_in(Kern k, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(cheb_tile)", __FILE__, __LINE__);
  return AGCN_OK;
}

static CtArgs base_args(const agcn_plan* plan, const float* L, int add_identity, int F, int K) {
  CtArgs a{};
  a.order = plan->d_order; a.n_nodes = plan->d_n; a.node_off = plan->d_node_off; a.lap_off = plan->d_lap_off;
  a.chunks = (F + CH - 1) / CH;
  a.L = L; a.add_identity = add_identity; a.F = F; a.K = K;
  return a;
}

// the bucket of graphs between AGCN_FUSE_MAX_N and AGCN_SMALL_MAX nodes that run per-graph (not row-tiled), or NULL
static const Bucket* mid_bucket(const agcn_plan* plan) {
  for (const Bucket& b : plan->buckets)
    if (b.limit > AGCN_FUSE_MAX_N && b.max_n <= plan->cheb_small_max) return &b;
  return nullptr;
}

static int launch(const agcn_plan* plan, CtArgs a, bool forward, cudaStream_t st_small, cudaStream_t st_mid) {
  static std::once_flag once;
  static int once_rc = AGCN_OK;
  const size_t smem_tile = smem_bytes(128, AGCN_FUSE_LCAP, true);
  const int mid_rows = (AGCN_SMALL_MAX + 31) / 32 * 32;
  const size_t smem_mid = smem_bytes(mid_rows, AGCN_SMALL_MAX * (AGCN_SMALL_MAX | 1), false);
  std::call_once(once, [&] {
    int rc;
    if ((rc = opt_in(cheb_tile_fwd_kernel<true, 2>, smem_tile))) once_rc = rc;
    if ((rc = opt_in(cheb_tile_bwd_kernel<true, 2>, smem_tile))) once_rc = rc;
    if ((rc = opt_in(cheb_tile_fwd_kernel<false, 5>, smem_mid))) once_rc = rc;
    if ((rc = opt_in(cheb_tile_bwd_kernel<false, 5>, smem_mid))) once_rc = rc;
  });
  if (once_rc) return once_rc;
  // the mid-size graphs first: each needs most of an SM's shared memory and would otherwise queue behind the tile CTAs
  if (const Bucket* b = mid_bucket(plan)) {
    CtArgs t = a;
    t.tile_graphs = nullptr;
    t.order_start = b->start;
    t.rows = mid_rows;
    t.lfloats = AGCN_SMALL_MAX * (AGCN_SMALL_MAX | 1);
    t.cpc = 1;
    t.groups = t.chunks;
    const unsigned grid = (unsigned)(b->count * t.chunks);
    {
      ProfScope prof(forward ? "ct::cheb_tile_fwd_kernel(mid)" : "ct::cheb_tile_bwd_kernel(mid)", st_mid);
      if (forward)
        cheb_tile_fwd_kernel<false, 5><<<grid, 2 * mid_rows, smem_mid, st_mid>>>(t);
      else
        cheb_tile_bwd_kernel<false, 5><<<grid, 2 * mid_rows, smem_mid, st_mid>>>(t);
    }
    AGCN_LAUNCH_CHECK();
  }
  if (plan->ft_small_tiles > 0) {
    CtArgs t = a;
    t.tile_graphs = reinterpret_cast<const int4*>(plan->d_ft_entries);
    t.tile_gstart = plan->d_ft_gstart;
    t.rows = 128;
    t.lfloats = AGCN_FUSE_LCAP;
    // chunks per CTA: the smallest count that makes the grid ONE wave of the 3 CTAs per SM (the prologue -- graph list,
    // L matrices, masks: 5 of a CTA's 11 us -- is paid once per CTA, and a partial second wave costs a whole one)
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    t.cpc = 1;
    while (t.cpc < t.chunks && plan->ft_small_tiles * ((t.chunks + t.cpc - 1) / t.cpc) > 3 * sms) ++t.cpc;
    t.groups = (t.chunks + t.cpc - 1) / t.cpc;
    const unsigned grid = (unsigned)(plan->ft_small_tiles * t.groups);
    ProfScope prof(forward ? "ct::cheb_tile_fwd_kernel" : "ct::cheb_tile_bwd_kernel", st_small);
    if (forward)
      cheb_tile_fwd_kernel<true, 2><<<grid, 256, smem_tile, st_small>>>(t);
    else
      cheb_tile_bwd_kernel<true, 2><<<grid, 256, smem_tile, st_small>>>(t);
  }
  if (plan->ft_small_tiles > 0) AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // namespace ct

bool cheb_tiles_has_mid(const agcn_plan* plan) { return ct::mid_bucket(plan) != nullptr; }

// T_1 .. T_{K-1} of every graph up to AGCN_SMALL_MAX nodes that is not row-tiled (small-graph tiles on st_small, the
// mid-size graphs on st_mid)
int cheb_tiles_forward(const agcn_plan* plan, const float* X, const float* L, int add_identity, int F, int K, float* T,
                       cudaStream_t st_small, cudaStream_t st_mid, int transL) {
  if (K < 2) return AGCN_OK;
  ct::CtArgs a = ct::base_args(plan, L, add_identity, F, K);
  a.transL = transL;
  a.X = X; a.T = T; a.tslice = (long long)plan->R * F;
  return ct::launch(plan, a, true, st_small, st_mid);
}

// dX rows of the same graphs from G_z = dYpre W_z^T
int cheb_tiles_backward(const agcn_plan* plan, const float* G, const float* L, int add_identity, int F, int K, float* dX,
                        cudaStream_t st_small, cudaStream_t st_mid) {
  if (K < 2) return AGCN_OK;
  ct::CtArgs a = ct::base_args(plan, L, add_identity, F, K);
  a.G = G; a.gslice = (long long)plan->R * F; a.dX = dX;
  return ct::launch(plan, a, false, st_small, st_mid);
}

}  // namespace agcn
