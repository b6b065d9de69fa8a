// Chebyshev products of the graphs that do not fit the fused tile kernels (n > cheb_small_max: point clouds,
// ModelNet40-shape N = 1024, Sydney-shape ragged N, the N <= 4096 sweep), on the tensor cores:
//
//     Out = cmul * op(L_g) * In  (+ Add)  (- Sub)  (+ RowScale .* ScaleIn),    op(L) = L (+ I) | L^T (+ I)
//
// forward T_k = 2 L T_{k-1} - T_{k-2} (graphconv.py:221-236), its reverse recurrence U_j = G_j + c L^T U_{j+1} - U_{j+2},
// and the dXW = rowsum(C) xw - C XW product of the metric gradient.  At n = 1024, F = 128 one step is a
// [1024 x 1024] x [1024 x 128] contraction per graph: dense tensor-core work (north_star item 3).
//
// grouped_tc_kernel: one CTA per (graph, 128-row tile, 128-column block of the node matrix).
//   warps 2-17: A = L_g[rows, k-block of 32 columns] loaded from global memory (ragged n: rows are not 16-byte
//               aligned, so no TMA), split into hi / lo TF32 halves and written as a 128 x 32 K-major SWIZZLE_128B
//               operand (transposed on the fly for L^T); the B tile brought by TMA is split in place;
//   warp 0    : TMA producer of B = In[k-block of 32 nodes, 128 columns]: row-major node matrix = MN-major operand,
//               32 x 32 boxes in the 128B-swizzle / 32B-atom layout (as in tc_gemm_tn_kernel);
//   warp 1    : tcgen05.mma kind::tf32, 3xTF32 (A_lo B_hi + A_hi B_lo + A_hi B_hi) into a TMEM accumulator;
//   epilogue  : TMEM -> registers -> shared -> coalesced float4 rows with the recurrence terms applied.
// Rows of In that belong to the next graph (last k-block of a ragged graph) are zeroed during the split, so a
// non-finite value never crosses a graph boundary.
//
// grouped_thin_kernel{,_t}: the 3- or 4-feature first layer of a point cloud (F <= 8) is a stream over L with
// 2 F flop per element: plain fp32 FMAs, L read once with coalesced rows (columns for L^T).
#include <cuda.h>

#include <algorithm>
#include <mutex>

#include "agcn_internal.cuh"

namespace agcn {
namespace bt {

constexpr int TM = 128;
constexpr int BK = 32;
constexpr int UMMA_K = 8;
constexpr int BN = 128;                     // node-matrix columns per CTA
constexpr int A_BYTES = TM * BK * 4;        // 16 KB: one half (hi or lo) of the A operand of a k-block
constexpr int B_BYTES = BN * BK * 4;        // 16 KB: four 32 x 32 boxes
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
constexpr int STAGES = 3;
constexpr int WORKERS = 512;            // 16 worker warps: the operand split is a latency chain per warp
constexpr int NW = WORKERS / 32;
constexpr int AHEAD = 4;                // k-blocks of L in flight per thread (register prefetch)
constexpr int CPT = 1024 / WORKERS;     // 16-byte chunks of the A tile (and float4s of a full B tile) per thread and k-block
constexpr int THREADS = 64 + WORKERS;
constexpr int SMEM_TOTAL = STAGES * STAGE_BYTES + 256 + 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait_shared(smem_u32(bar), parity); }
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// A: K-major, SWIZZLE_128B, 8-row atoms of 1024 bytes (same operand format as agcn_pre_tile.cu)
__device__ __forceinline__ uint64_t make_desc_k(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// B: MN-major TF32, 128B swizzle with 32B atoms (same operand format as tc_gemm_tn_kernel): 32-column groups
// 4096 bytes apart, groups of 4 contraction rows 512 bytes apart
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(4096 >> 4) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float v[32]) {
  uint32_t u[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
      "%29,%30,%31}, [%32];\n"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
        "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
        "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void sts32(uint32_t a, float v) {
  asm volatile("st.shared.f32 [%0], %1;\n" ::"r"(a), "f"(v) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};\n" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float tf32_hi(float x) { return tf32_rn(x); }
__device__ __forceinline__ float tf32_lo(float x, float hi) { return tf32_rn(x - hi); }

__global__ void __launch_bounds__(THREADS, 1)
grouped_tc_kernel(const __grid_constant__ CUtensorMap tmIn, GroupedArgs p) {
  const int g = p.tile_graph[blockIdx.x], m0 = p.tile_row[blockIdx.x];
  if (m0 & (TM - 1)) return;  // the plan lists 64-row tiles: every even one starts a 128-row tile of this kernel
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(base);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + STAGES * STAGE_BYTES);
  uint64_t* full_bar = bars;              // B tile landed (TMA)
  uint64_t* split_bar = bars + STAGES;    // A written and B split by the worker warps
  uint64_t* empty_bar = bars + 2 * STAGES;  // MMAs that read the stage retired
  uint64_t* tmem_full_bar = bars + 3 * STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = p.n_nodes[g];
  const long long row0 = p.node_off[g];
  const float* __restrict__ Lg = p.L + p.lap_off[g];
  const int F = p.F;
  const int f0 = blockIdx.y * BN;
  const int b_boxes = min(BN / 32, (F - f0 + 31) / 32);
  const int nmma = 32 * b_boxes;
  const int num_kb = (n + BK - 1) / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&split_bar[s], WORKERS / 32);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;\n" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int stage = kb % STAGES, phase = (kb / STAGES) & 1;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        const uint32_t sb = sbase + stage * STAGE_BYTES + 2 * A_BYTES;
        mbar_expect_tx(&full_bar[stage], b_boxes * 4096);
        for (int b = 0; b < b_boxes; ++b)
          tma_load_2d(sb + b * 4096, &tmIn, &full_bar[stage], f0 + 32 * b, (int)(row0 + (long long)kb * BK));
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // D = f32, A = tf32 K-major, B = tf32 MN-major, N = nmma, M = 128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)(nmma >> 3) << 17) |
                             ((uint32_t)(TM >> 4) << 24);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int stage = kb % STAGES, phase = (kb / STAGES) & 1;
        mbar_wait(&split_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = sbase + stage * STAGE_BYTES, sa_lo = sa + A_BYTES;
        const uint32_t sb = sa + 2 * A_BYTES, sb_lo = sb + B_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t a_hi = make_desc_k(sa + k * UMMA_K * 4), a_lo = make_desc_k(sa_lo + k * UMMA_K * 4);
          const uint64_t b_hi = make_desc_mn(sb + k * 1024), b_lo = make_desc_mn(sb_lo + k * 1024);
          umma_tf32(tmem_base, a_lo, b_hi, idesc, (kb | k) != 0);
          umma_tf32(tmem_base, a_hi, b_lo, idesc, 1);
          umma_tf32(tmem_base, a_hi, b_hi, idesc, 1);
        }
        umma_commit(&empty_bar[stage]);
      }
      umma_commit(tmem_full_bar);
    }
  } else {
    const int ww = warp - 2;              // worker warp 0..NW-1
    const int wt = ww * 32 + lane;
    // ---- A loader: every thread owns four 16-byte chunks (4 consecutive contraction columns of one operand row) per
    // k-block, so the split costs one 128-bit shared store per chunk and half.
    //   op = L  : 8 lanes cover the 32 columns of a row (a float4 each when the graph's rows are 16-byte aligned), a
    //             warp covers rows (128 / NW) ww + 4 t + lane / 8;
    //   op = L^T: warp ww owns chunk ww % 8 (contraction rows 4 c .. 4 c + 3 of the k-block) of the operand rows
    //             (ww / 8) * 32 CPT + 32 t + lane: four coalesced scalar loads along a row of L fill the chunk.
    // Either way the 32 lanes of a store hit 4 x 8 distinct 16-byte slots of the swizzled tile: no bank conflicts.
    const bool vecL = !p.transL && ((n & 3) == 0) && ((reinterpret_cast<uintptr_t>(Lg) & 15) == 0);
    // per-thread constants of its CPT chunks: operand row, swizzled byte offset in the tile, global address at k-block 0
    int arow[CPT];
    uint32_t aoff[CPT];
    const float* aptr[CPT];
#pragma unroll
    for (int t = 0; t < CPT; ++t) {
      const int r = p.transL ? (ww >> 3) * (32 * CPT) + 32 * t + lane : ww * (TM / NW) + 4 * t + (lane >> 3);
      const int chunk = p.transL ? (ww & 7) : (lane & 7);
      arow[t] = r;
      aoff[t] = (uint32_t)(r * 128 + ((chunk ^ (r & 7)) << 4));
      aptr[t] = p.transL ? Lg + (long long)(4 * chunk) * n + (m0 + r) : Lg + (long long)(m0 + r) * n + 4 * chunk;
    }
    // interior k-blocks of a tile whose 128 rows all exist need no bounds checks (every k-block of a point cloud with
    // n % 128 == 0); op = L additionally wants 16-byte aligned rows for the float4 loads
    const bool fast_rows = (m0 + TM <= n) && (p.transL || vecL);
    const long long kstep = p.transL ? (long long)BK * n : BK;   // elements between consecutive k-blocks
    auto load_a = [&](int kb, float4 (&v)[CPT]) {
      if (kb >= num_kb) return;
      const int k0 = kb * BK;
      if (fast_rows && k0 + BK <= n) {
#pragma unroll
        for (int t = 0; t < CPT; ++t) {
          const float* src = aptr[t] + kb * kstep;
          if (!p.transL) {
            v[t] = __ldg(reinterpret_cast<const float4*>(src));
          } else {
            v[t].x = __ldg(src);
            v[t].y = __ldg(src + n);
            v[t].z = __ldg(src + 2 * (long long)n);
            v[t].w = __ldg(src + 3 * (long long)n);
          }
        }
        return;
      }
#pragma unroll
      for (int t = 0; t < CPT; ++t) {
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        const int i = m0 + arow[t];
        const float* src = aptr[t] + kb * kstep;
        if (!p.transL) {
          const int j = k0 + 4 * (lane & 7);
          if (i < n && j < n) {
            if (vecL) {
              x = __ldg(reinterpret_cast<const float4*>(src));
            } else {
              x.x = __ldg(src);
              if (j + 1 < n) x.y = __ldg(src + 1);
              if (j + 2 < n) x.z = __ldg(src + 2);
              if (j + 3 < n) x.w = __ldg(src + 3);
            }
          }
        } else {
          const int j = k0 + 4 * (ww & 7);
          if (i < n && j < n) {
            x.x = __ldg(src);
            if (j + 1 < n) x.y = __ldg(src + n);
            if (j + 2 < n) x.z = __ldg(src + 2 * (long long)n);
            if (j + 3 < n) x.w = __ldg(src + 3 * (long long)n);
          }
        }
        v[t] = x;
      }
    };
    auto split_store = [&](uint32_t a_hi, uint32_t a_lo, const float4& x) {
      float4 hi, lo;
      hi.x = tf32_hi(x.x); hi.y = tf32_hi(x.y); hi.z = tf32_hi(x.z); hi.w = tf32_hi(x.w);
      lo.x = tf32_lo(x.x, hi.x); lo.y = tf32_lo(x.y, hi.y); lo.z = tf32_lo(x.z, hi.z); lo.w = tf32_lo(x.w, hi.w);
      sts128(a_hi, hi);
      sts128(a_lo, lo);
    };
    // B: float4 number idx = wt + WORKERS t of the landed tile (256 per 32-column box); which of mine exist
    bool bmine[CPT];
    int bkrow[CPT];
#pragma unroll
    for (int t = 0; t < CPT; ++t) {
      const int idx = wt + WORKERS * t;
      bmine[t] = idx < b_boxes * 256;
      bkrow[t] = (idx & 255) >> 3;   // contraction row of the k-block this float4 belongs to
    }
    auto step = [&](int kb, float4 (&v)[CPT]) {
      const int stage = kb % STAGES, phase = (kb / STAGES) & 1;
      const uint32_t st = sbase + stage * STAGE_BYTES;
      if (lane == 0) mbar_wait(&empty_bar[stage], phase ^ 1);
      __syncwarp();
#pragma unroll
      for (int t = 0; t < CPT; ++t) split_store(st + aoff[t], st + A_BYTES + aoff[t], v[t]);
      load_a(kb + AHEAD, v);             // AHEAD k-blocks ahead of their use
      mbar_wait(&full_bar[stage], phase);  // every lane: the TMA bytes are read right below
      const int valid = n - kb * BK;     // contraction rows of this k-block that belong to the graph
      const uint32_t sb = st + 2 * A_BYTES + 16 * wt;
      float4 x[CPT];
#pragma unroll
      for (int t = 0; t < CPT; ++t) {      // every load first: the chunks are independent
        x[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (bmine[t] && bkrow[t] < valid) x[t] = lds128(sb + 16 * WORKERS * t);
      }
#pragma unroll
      for (int t = 0; t < CPT; ++t)
        if (bmine[t]) split_store(sb + 16 * WORKERS * t, sb + 16 * WORKERS * t + B_BYTES, x[t]);
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) mbar_arrive(&split_bar[stage]);
    };
    float4 va[CPT], vb[CPT], vc[CPT], vd[CPT];   // AHEAD register buffers, one per k-block in flight
    load_a(0, va);
    load_a(1, vb);
    load_a(2, vc);
    load_a(3, vd);
    for (int kb = 0; kb < num_kb; kb += AHEAD) {
      step(kb, va);
      if (kb + 1 < num_kb) step(kb + 1, vb);
      if (kb + 2 < num_kb) step(kb + 2, vc);
      if (kb + 3 < num_kb) step(kb + 3, vd);
    }
    // ---- epilogue
    if (lane == 0) mbar_wait(tmem_full_bar, 0);
    __syncwarp();
    tc_fence_after();
    const int q = warp & 3;      // TMEM lane quarter of this warp
    const int h = ww >> 2;       // 32-column group of this warp (NW / 4 groups)
    // The operand stages are free now: the accumulator barrier fires after the last MMA, which waited for every warp's
    // operand stores.  The named barrier says so in a form compute-sanitizer's racecheck understands (it does not follow
    // mbarrier / tcgen05.commit ordering and reported the staging stores against the other warps' operand stores).
    asm volatile("bar.sync 1, %0;\n" ::"n"(WORKERS) : "memory");
    const uint32_t stg = sbase + (uint32_t)(ww * (32 * 36 * 4));
    for (int c0 = 32 * h; c0 < nmma; c0 += 32 * (NW / 4)) {
      float v[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        sts128(stg + 4 * (lane * 36 + 4 * u), make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]));
      __syncwarp();
      const int c = f0 + c0 + 4 * (lane & 7);
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int rr = 4 * t + (lane >> 3);
        const int i = m0 + q * 32 + rr;
        if (i >= n || c >= F) continue;  // F % 4 == 0: a float4 is inside or outside as a whole
        const float4 a4 = lds128(stg + 4 * (rr * 36 + 4 * (lane & 7)));
        const long long o = (row0 + i) * F + c;
        float4 r4 = make_float4(p.cmul * a4.x, p.cmul * a4.y, p.cmul * a4.z, p.cmul * a4.w);
        if (p.add_identity) {  // (L + I) In = L In + In
          const float4 x = *reinterpret_cast<const float4*>(p.In + o);
          r4.x = fmaf(p.cmul, x.x, r4.x); r4.y = fmaf(p.cmul, x.y, r4.y);
          r4.z = fmaf(p.cmul, x.z, r4.z); r4.w = fmaf(p.cmul, x.w, r4.w);
        }
        if (p.Add) {
          const float4 x = *reinterpret_cast<const float4*>(p.Add + o);
          r4.x += x.x; r4.y += x.y; r4.z += x.z; r4.w += x.w;
        }
        if (p.Sub) {
          const float4 x = *reinterpret_cast<const float4*>(p.Sub + o);
          r4.x -= x.x; r4.y -= x.y; r4.z -= x.z; r4.w -= x.w;
        }
        if (p.RowScale) {
          const float sc = p.RowScale[row0 + i];
          const float4 x = *reinterpret_cast<const float4*>(p.ScaleIn + o);
          r4.x = fmaf(sc, x.x, r4.x); r4.y = fmaf(sc, x.y, r4.y); r4.z = fmaf(sc, x.z, r4.z); r4.w = fmaf(sc, x.w, r4.w);
        }
        *reinterpret_cast<float4*>(p.Out + o) = r4;
        if (p.Out2) *reinterpret_cast<float4*>(p.Out2 + o) = r4;
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;\n" ::"r"(tmem_base) : "memory");
}

// ------------------------------------------------------------------------------------------------
// grouped_tcu_kernel: the same product for batches of EQUAL-SIZE graphs with n % 128 == 0 (ModelNet40-shape point clouds,
// the N >= 128 sweep points), where every row of L is 16-byte aligned and L is one [B n, n] matrix for TMA.
//
// grouped_tc_kernel above loads its L tiles with register prefetch four k-blocks ahead -- and ends every k-block with
// fence.proxy.async, which ptxas lowers to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC: the MEMBAR waits for every load the thread
// has in flight, so the prefetch never overlapped anything (1.05 us per k-block against 0.55 us of MMA work, 12 % of the
// TF32 peak; profiles/r01_n_tc_timeline_3stage.txt).  Here, as in pt::rows_gemm_kernel:
//   * raw fp32 L tiles arrive by TMA (128 rows x 32 columns SWIZZLE_128B; for L^T the 32 x 128 block of L, unswizzled,
//     read column-wise -- the transposition costs nothing) from their own producer thread;
//   * the workers split a staged tile into hi / lo TF32 halves and write them into an operand slot in TENSOR MEMORY
//     (tcgen05.st): the MMAs take A from TMEM, shared memory serves only the node-matrix operand;
//   * the node-matrix tile (MN-major, by TMA) is split in place as before; the proxy fence behind it is cheap now that
//     no global load is outstanding in the fencing threads;
//   * two CTAs per SM (256 TMEM columns, ~100 KB of shared memory each): 256 row tiles of a 32-cloud batch are one wave.
// ------------------------------------------------------------------------------------------------
constexpr int U_THREADS = 96 + 256;   // warp 0: node-matrix tiles, warp 1: MMA, warp 2: L tiles, warps 3..10 workers
constexpr int U_NB = 2, U_NS = 2, U_NA = 2;
constexpr int U_CTAS = 2, U_TMEM = 256;   // measured at C3 (32 x 1024 points, F = 128): 71 us per product; one CTA per SM with
                                          // 4 / 4 / 3-deep rings and 512 TMEM columns: 93 us (256 tiles are then two waves)
constexpr int U_SMEM = U_NB * 2 * B_BYTES + U_NS * A_BYTES + 256 + 1024;

__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float v[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];\n" : "=f"(v) : "r"(a) : "memory");
  return v;
}

__global__ void __launch_bounds__(U_THREADS, U_CTAS)
grouped_tcu_kernel(const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmL, GroupedArgs p, int n) {
  const int g = p.tile_graph[blockIdx.x], m0 = p.tile_row[blockIdx.x];
  if (m0 & (TM - 1)) return;  // the plan lists 64-row tiles: every even one starts a 128-row tile of this kernel
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(base);
  const uint32_t b_ring = sbase, s_ring = sbase + U_NB * 2 * B_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + U_NB * 2 * B_BYTES + U_NS * A_BYTES);
  uint64_t* b_full = bars;         // [NB] node-matrix tile landed (TMA)
  uint64_t* b_split = bars + 4;    // [NB] ... and split in place by the 8 worker warps
  uint64_t* b_empty = bars + 8;    // [NB] the MMAs that read it retired
  uint64_t* s_full = bars + 12;    // [NS] raw L tile landed (TMA)
  uint64_t* s_empty = bars + 16;   // [NS] the 8 worker warps have read it
  uint64_t* a_full = bars + 20;    // [NA] operand slot in tensor memory written
  uint64_t* a_empty = bars + 24;   // [NA] the MMAs that read the slot retired
  uint64_t* out_bar = bars + 28;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 29);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row0 = (long long)g * n;   // equal-size graphs: node_off[g] = g n, lap_off[g] = g n^2
  const int F = p.F;
  const int f0 = blockIdx.y * BN;
  const int b_boxes = min(BN / 32, (F - f0 + 31) / 32);
  const int nmma = 32 * b_boxes;
  const int num_kb = n / BK;
  constexpr int A_COL0 = 128;   // operand slots behind the accumulator: slot s = [hi 32 | lo 32] columns

  if (threadIdx.x == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(&b_full[s], 1);
      mbar_init(&b_split[s], 8);
      mbar_init(&b_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], 8);
      mbar_init(&a_full[s], 8);
      mbar_init(&a_empty[s], 1);
    }
    mbar_init(out_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "n"(U_TMEM) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int slot = kb % U_NB, u = kb / U_NB;
        if (u > 0) mbar_wait(&b_empty[slot], (uint32_t)((u - 1) & 1));
        const uint32_t sb = b_ring + slot * 2 * B_BYTES;
        mbar_expect_tx(&b_full[slot], b_boxes * 4096);
        for (int b = 0; b < b_boxes; ++b)
          tma_load_2d(sb + b * 4096, &tmIn, &b_full[slot], f0 + 32 * b, (int)(row0 + (long long)kb * BK));
      }
    }
  } else if (warp == 2) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int slot = kb % U_NS, u = kb / U_NS;
        if (u > 0) mbar_wait(&s_empty[slot], (uint32_t)((u - 1) & 1));
        mbar_expect_tx(&s_full[slot], A_BYTES);
        if (!p.transL)   // rows m0.. of L_g, columns of the k-block
          tma_load_2d(s_ring + slot * A_BYTES, &tmL, &s_full[slot], kb * BK, (int)(row0 + m0));
        else             // rows of the k-block of L_g, columns m0..: read column-wise by the workers
          tma_load_2d(s_ring + slot * A_BYTES, &tmL, &s_full[slot], m0, (int)(row0 + (long long)kb * BK));
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // D = f32, A = tf32 from tensor memory, B = tf32 MN-major, N = nmma, M = 128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)(nmma >> 3) << 17) |
                             ((uint32_t)(TM >> 4) << 24);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int aslot = kb % U_NA, bslot = kb % U_NB;
        mbar_wait(&a_full[aslot], (uint32_t)((kb / U_NA) & 1));
        mbar_wait(&b_split[bslot], (uint32_t)((kb / U_NB) & 1));
        tc_fence_after();
        const uint32_t ta_hi = tmem_base + (uint32_t)(A_COL0 + aslot * 2 * BK), ta_lo = ta_hi + BK;
        const uint32_t sb = b_ring + bslot * 2 * B_BYTES, sb_lo = sb + B_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t b_hi = make_desc_mn(sb + k * 1024), b_lo = make_desc_mn(sb_lo + k * 1024);
          umma_ts(tmem_base, ta_lo + k * UMMA_K, b_hi, idesc, (kb | k) != 0);
          umma_ts(tmem_base, ta_hi + k * UMMA_K, b_lo, idesc, 1);
          umma_ts(tmem_base, ta_hi + k * UMMA_K, b_hi, idesc, 1);
        }
        umma_commit(&b_empty[bslot]);
        umma_commit(&a_empty[aslot]);
      }
      umma_commit(out_bar);
    }
  } else {
    const int wi = warp - 3, q = warp & 3, h = wi >> 2, r = q * 32 + lane;
    const int wt = wi * 32 + lane;
    uint32_t soff[4];
#pragma unroll
    for (int gq = 0; gq < 4; ++gq) soff[gq] = (uint32_t)(r * 128 + (((4 * h + gq) ^ (r & 7)) << 4));
    for (int kb = 0; kb < num_kb; ++kb) {
      const int sslot = kb % U_NS, aslot = kb % U_NA, bslot = kb % U_NB;
      // ---- A: staged raw L tile -> hi / lo halves of my 16 contraction columns in my TMEM lane
      if (lane == 0) {
        mbar_wait(&s_full[sslot], (uint32_t)((kb / U_NS) & 1));
        if (kb >= U_NA) mbar_wait(&a_empty[aslot], (uint32_t)((kb / U_NA - 1) & 1));
      }
      __syncwarp();
      const uint32_t st = s_ring + sslot * A_BYTES;
      float x[16];
      if (!p.transL) {
#pragma unroll
        for (int gq = 0; gq < 4; ++gq) {
          const float4 v = lds128(st + soff[gq]);
          x[4 * gq] = v.x; x[4 * gq + 1] = v.y; x[4 * gq + 2] = v.z; x[4 * gq + 3] = v.w;
        }
      } else {
#pragma unroll
        for (int u = 0; u < 16; ++u) x[u] = lds32(st + (uint32_t)((16 * h + u) * (TM * 4) + r * 4));   // L[k0 + 16h + u][m0 + r]
      }
      float hi[16], lo[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        hi[u] = tf32_hi(x[u]);
        lo[u] = tf32_lo(x[u], hi[u]);
      }
      const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(A_COL0 + aslot * 2 * BK + 16 * h);
      tmem_st16(ta, hi);
      tmem_st16(ta + BK, lo);
      asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&s_empty[sslot]);
        mbar_arrive(&a_full[aslot]);
      }
      // ---- B: split the landed node-matrix tile in place
      mbar_wait(&b_full[bslot], (uint32_t)((kb / U_NB) & 1));   // every lane: the TMA bytes are read right below
      const uint32_t sb = b_ring + bslot * 2 * B_BYTES + 16 * wt;
      float4 y[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        y[t] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (wt + 256 * t < b_boxes * 256) y[t] = lds128(sb + 16 * 256 * t);
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        if (wt + 256 * t < b_boxes * 256) {
          float4 bh, bl;
          bh.x = tf32_hi(y[t].x); bh.y = tf32_hi(y[t].y); bh.z = tf32_hi(y[t].z); bh.w = tf32_hi(y[t].w);
          bl.x = tf32_lo(y[t].x, bh.x); bl.y = tf32_lo(y[t].y, bh.y); bl.z = tf32_lo(y[t].z, bh.z); bl.w = tf32_lo(y[t].w, bh.w);
          sts128(sb + 16 * 256 * t, bh);
          sts128(sb + 16 * 256 * t + B_BYTES, bl);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) mbar_arrive(&b_split[bslot]);
    }
    // ---- epilogue
    if (lane == 0) mbar_wait(out_bar, 0);
    __syncwarp();
    tc_fence_after();
    __syncwarp();
    asm volatile("bar.sync 1, 256;\n" ::: "memory");   // every worker is past its last tile before the rings are reused
    const uint32_t stg = sbase + (uint32_t)(wi * (32 * 36 * 4));
    for (int c0 = 32 * h; c0 < nmma; c0 += 64) {
      float v[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
      for (int u = 0; u < 8; ++u)
        sts128(stg + 4 * (lane * 36 + 4 * u), make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]));
      __syncwarp();
      const int c = f0 + c0 + 4 * (lane & 7);
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        const int rr = 4 * t + (lane >> 3);
        const int i = m0 + q * 32 + rr;
        if (c >= F) continue;  // F % 4 == 0: a float4 is inside or outside as a whole
        const float4 a4 = lds128(stg + 4 * (rr * 36 + 4 * (lane & 7)));
        const long long o = (row0 + i) * F + c;
        float4 r4 = make_float4(p.cmul * a4.x, p.cmul * a4.y, p.cmul * a4.z, p.cmul * a4.w);
        if (p.add_identity) {  // (L + I) In = L In + In
          const float4 xx = *reinterpret_cast<const float4*>(p.In + o);
          r4.x = fmaf(p.cmul, xx.x, r4.x); r4.y = fmaf(p.cmul, xx.y, r4.y);
          r4.z = fmaf(p.cmul, xx.z, r4.z); r4.w = fmaf(p.cmul, xx.w, r4.w);
        }
        if (p.Add) {
          const float4 xx = *reinterpret_cast<const float4*>(p.Add + o);
          r4.x += xx.x; r4.y += xx.y; r4.z += xx.z; r4.w += xx.w;
        }
        if (p.Sub) {
          const float4 xx = *reinterpret_cast<const float4*>(p.Sub + o);
          r4.x -= xx.x; r4.y -= xx.y; r4.z -= xx.z; r4.w -= xx.w;
        }
        if (p.RowScale) {
          const float sc = p.RowScale[row0 + i];
          const float4 xx = *reinterpret_cast<const float4*>(p.ScaleIn + o);
          r4.x = fmaf(sc, xx.x, r4.x); r4.y = fmaf(sc, xx.y, r4.y); r4.z = fmaf(sc, xx.z, r4.z); r4.w = fmaf(sc, xx.w, r4.w);
        }
        *reinterpret_cast<float4*>(p.Out + o) = r4;
        if (p.Out2) *reinterpret_cast<float4*>(p.Out2 + o) = r4;
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(U_TMEM) : "memory");
}

// ------------------------------------------------------------------------------------------------
// pair_tcu_kernel: 128 x 128 tiles of the n x n PAIR matrices of big equal-size graphs on the tensor cores (the learned
// metric of graphconv.py:163-209 and its gradient; north_star item 1):
//
//   SIM   gram_ij = <xw_i, xw_j>  ->  dist_ij = sqrt(|xw_i|^2 + |xw_j|^2 - 2 gram_ij),  W_ij = exp(-dist_ij), W_ii = 0,
//         row sums of W per 64-column block (the degree vector)                              graphconv.py:171-178,195
//   DL    dL_ij = dLall_in_ij + sum_{s} c_s <U_s[i, :], T_{s-1}[j, :]>                        (reverse mode of :231-234)
//
// Both operands are K-major row panels of node matrices ([128 nodes x 32 features], raw fp32 by TMA): the i panel is
// split into hi / lo TF32 halves into an operand slot in tensor memory, the j panel in place in shared memory (3xTF32).
// SIM: the Gram expansion cancels for near-duplicate rows (SURVEY Q7): an entry whose Gram error (~1e-6 of the norms)
// would move W = exp(-dist) or the metric gradient by more than 1e-5 is recomputed from direct differences in fp32 --
// the nearest neighbours of a point; far pairs (W ~ 0) never are.  The SIMT kernel this replaces (big_pair_kernel, 64 x 64 tiles of direct
// differences / FMAs) took 290 us (SIM) and 410 us (DL) per layer at 32 x 1024 points, F = 128.
// ------------------------------------------------------------------------------------------------
struct PairTcArgs {
  const int32_t* tile_graph;
  const int32_t* tile_row;
  int n, R, F, S, mode;          // mode 0 = SIM, 1 = DL; S = slices summed (SIM: 1)
  const float* dL_in;            // DL, optional
  float* out;                    // DL: dL
  const float* XW;               // SIM: the node matrix itself (fix-up) ...
  const float* mu;               //      [B][F] per-graph mean row: the Gram runs on CENTERED rows (distances do not change,
                                 //      the norms shrink to the spread of the cloud, so the expansion cancels far less)
  const float* norms;            //      |xw_i - mu|^2 per packed row
  float* dist;                   //      optional
  float* resW;                   //      optional
  float* rowpart;                //      optional [R][ncb] row sums of W per 64-column block
  int ncb;
};

template <bool DL>
__global__ void __launch_bounds__(U_THREADS, 2)
pair_tcu_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB0,
                const __grid_constant__ CUtensorMap tmB1, PairTcArgs p) {
  const int g = p.tile_graph[blockIdx.x], m0 = p.tile_row[blockIdx.x];
  if (m0 & (TM - 1)) return;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(base);
  const uint32_t b_ring = sbase, s_ring = sbase + U_NB * 2 * B_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + U_NB * 2 * B_BYTES + U_NS * A_BYTES);
  uint64_t* b_full = bars;
  uint64_t* b_split = bars + 4;
  uint64_t* b_empty = bars + 8;
  uint64_t* s_full = bars + 12;
  uint64_t* s_empty = bars + 16;
  uint64_t* a_full = bars + 20;
  uint64_t* a_empty = bars + 24;
  uint64_t* out_bar = bars + 28;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 29);
  const uint32_t s_mu = sbase + U_NB * 2 * B_BYTES + U_NS * A_BYTES + 256;   // F floats (SIM)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = p.n, F = p.F, nc = F / BK;
  const long long row0 = (long long)g * n;
  const int j0 = blockIdx.y * TM;
  const int num_kb = p.S * nc;
  constexpr int A_COL0 = 128;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(&b_full[s], 1);
      mbar_init(&b_split[s], 8);
      mbar_init(&b_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], 8);
      mbar_init(&a_full[s], 8);
      mbar_init(&a_empty[s], 1);
    }
    mbar_init(out_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;\n" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  for (int f = threadIdx.x; f < F; f += blockDim.x) sts32(s_mu + 4 * f, (!DL && p.mu) ? __ldg(p.mu + (long long)g * F + f) : 0.f);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {   // j panel: B_s = XW (SIM) | s == 0 ? X : T_s (DL)
      for (int kb = 0; kb < num_kb; ++kb) {
        const int slot = kb % U_NB, u = kb / U_NB;
        if (u > 0) mbar_wait(&b_empty[slot], (uint32_t)((u - 1) & 1));
        const int s = kb / nc, c = kb - s * nc;
        mbar_expect_tx(&b_full[slot], A_BYTES);
        if (s == 0)
          tma_load_2d(b_ring + slot * 2 * B_BYTES, &tmB0, &b_full[slot], c * BK, (int)(row0 + j0));
        else
          tma_load_2d(b_ring + slot * 2 * B_BYTES, &tmB1, &b_full[slot], c * BK, (int)((long long)(s - 1) * p.R + row0 + j0));
      }
    }
  } else if (warp == 2) {
    if (lane == 0) {   // i panel: A_s = XW (SIM) | U_{s+1} (DL: slice s + 1 of the G buffer)
      for (int kb = 0; kb < num_kb; ++kb) {
        const int slot = kb % U_NS, u = kb / U_NS;
        if (u > 0) mbar_wait(&s_empty[slot], (uint32_t)((u - 1) & 1));
        const int s = kb / nc, c = kb - s * nc;
        const long long arow = (DL ? (long long)(s + 1) * p.R : 0) + row0 + m0;
        mbar_expect_tx(&s_full[slot], A_BYTES);
        tma_load_2d(s_ring + slot * A_BYTES, &tmA, &s_full[slot], c * BK, (int)arow);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // D = f32, A = tf32 from tensor memory, B = tf32 K-major, N = 128, M = 128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TM >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int aslot = kb % U_NA, bslot = kb % U_NB;
        mbar_wait(&a_full[aslot], (uint32_t)((kb / U_NA) & 1));
        mbar_wait(&b_split[bslot], (uint32_t)((kb / U_NB) & 1));
        tc_fence_after();
        const uint32_t ta_hi = tmem_base + (uint32_t)(A_COL0 + aslot * 2 * BK), ta_lo = ta_hi + BK;
        const uint32_t sb = b_ring + bslot * 2 * B_BYTES, sb_lo = sb + B_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint64_t b_hi = make_desc_k(sb + k * UMMA_K * 4), b_lo = make_desc_k(sb_lo + k * UMMA_K * 4);
          umma_ts(tmem_base, ta_lo + k * UMMA_K, b_hi, idesc, (kb | k) != 0);
          umma_ts(tmem_base, ta_hi + k * UMMA_K, b_lo, idesc, 1);
          umma_ts(tmem_base, ta_hi + k * UMMA_K, b_hi, idesc, 1);
        }
        umma_commit(&b_empty[bslot]);
        umma_commit(&a_empty[aslot]);
      }
      umma_commit(out_bar);
    }
  } else {
    const int wi = warp - 3, q = warp & 3, h = wi >> 2, r = q * 32 + lane;
    const int wt = wi * 32 + lane;
    uint32_t soff[4];
#pragma unroll
    for (int gq = 0; gq < 4; ++gq) soff[gq] = (uint32_t)(r * 128 + (((4 * h + gq) ^ (r & 7)) << 4));
    int fc = -BK;   // first feature column of the k-block
    for (int kb = 0; kb < num_kb; ++kb) {
      const int sslot = kb % U_NS, aslot = kb % U_NA, bslot = kb % U_NB;
      const float coef = (DL && kb >= nc) ? 2.f : 1.f;   // c_1 = 1, c_k = 2 (DL)
      fc = fc + BK == F ? 0 : fc + BK;
      if (lane == 0) {
        mbar_wait(&s_full[sslot], (uint32_t)((kb / U_NS) & 1));
        if (kb >= U_NA) mbar_wait(&a_empty[aslot], (uint32_t)((kb / U_NA - 1) & 1));
      }
      __syncwarp();
      const uint32_t st = s_ring + sslot * A_BYTES;
      float hi[16], lo[16];
#pragma unroll
      for (int gq = 0; gq < 4; ++gq) {
        float4 v = lds128(st + soff[gq]);
        if (!DL) {
          const float4 m4 = lds128(s_mu + 4 * (fc + 16 * h + 4 * gq));
          v.x -= m4.x; v.y -= m4.y; v.z -= m4.z; v.w -= m4.w;
        }
        const float x[4] = {DL ? coef * v.x : v.x, DL ? coef * v.y : v.y, DL ? coef * v.z : v.z, DL ? coef * v.w : v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          hi[4 * gq + e] = tf32_hi(x[e]);
          lo[4 * gq + e] = tf32_lo(x[e], hi[4 * gq + e]);
        }
      }
      const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(A_COL0 + aslot * 2 * BK + 16 * h);
      tmem_st16(ta, hi);
      tmem_st16(ta + BK, lo);
      asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&s_empty[sslot]);
        mbar_arrive(&a_full[aslot]);
      }
      // j panel: split in place (the swizzled K-major layout is the same for the raw tile and both halves)
      mbar_wait(&b_full[bslot], (uint32_t)((kb / U_NB) & 1));
      const uint32_t sb = b_ring + bslot * 2 * B_BYTES + 16 * wt;
      float4 y[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        y[t] = lds128(sb + 16 * 256 * t);
        if (!DL) {
          // 16-byte slot idx of the swizzled tile: row idx / 8, logical chunk (idx % 8) ^ (row % 8)
          const int idx = wt + 256 * t, brow = idx >> 3, chunk = (idx & 7) ^ (brow & 7);
          const float4 m4 = lds128(s_mu + 4 * (fc + 4 * chunk));
          y[t].x -= m4.x; y[t].y -= m4.y; y[t].z -= m4.z; y[t].w -= m4.w;
        }
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float4 bh, bl;
        bh.x = tf32_hi(y[t].x); bh.y = tf32_hi(y[t].y); bh.z = tf32_hi(y[t].z); bh.w = tf32_hi(y[t].w);
        bl.x = tf32_lo(y[t].x, bh.x); bl.y = tf32_lo(y[t].y, bh.y); bl.z = tf32_lo(y[t].z, bh.z); bl.w = tf32_lo(y[t].w, bh.w);
        sts128(sb + 16 * 256 * t, bh);
        sts128(sb + 16 * 256 * t + B_BYTES, bl);
      }
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&b_split[bslot]);
    }
    // ---- epilogue: my row i = m0 + r, my 64 columns j0 + 64 h ..
    if (lane == 0) mbar_wait(out_bar, 0);
    __syncwarp();
    tc_fence_after();
    const int i = m0 + r;
    if (DL) {
      // every accumulator is complete: the rings are free.  Rows of 32 values go through a 32 x 36 block per warp so
      // that dL_in is read and dL written as whole 128-byte row segments
      const uint32_t stg = sbase + 1024 + (uint32_t)(wi * (32 * 36 * 4));
      // (the accumulator barrier already orders every warp's operand stores before this point -- the last MMA waited for
      // all of them; the named barrier states it in a form compute-sanitizer's racecheck can see)
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
      for (int cb = 0; cb < 2; ++cb) {
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(64 * h + 32 * cb), v);
        const long long tile0 = (long long)g * n * n + (long long)(m0 + q * 32) * n + j0 + 64 * h + 32 * cb;
#pragma unroll
        for (int u = 0; u < 8; ++u)
          sts128(stg + 4 * (lane * 36 + 4 * u), make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]));
        __syncwarp();
        float4 a4[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const long long o = tile0 + (long long)(4 * t + (lane >> 3)) * n + 4 * (lane & 7);
          a4[t] = p.dL_in ? __ldg(reinterpret_cast<const float4*>(p.dL_in + o)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const int rr = 4 * t + (lane >> 3);
          float4 o = lds128(stg + 4 * (rr * 36 + 4 * (lane & 7)));
          o.x += a4[t].x; o.y += a4[t].y; o.z += a4[t].z; o.w += a4[t].w;
          *reinterpret_cast<float4*>(p.out + tile0 + (long long)rr * n + 4 * (lane & 7)) = o;
        }
        __syncwarp();
      }
    } else {
      // every accumulator is complete: the rings are free.  Norms of the j tile and a 32 x 36 transposition buffer per warp
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
      const uint32_t s_nj = sbase;                                        // 128 floats
      const uint32_t stg = sbase + 1024 + (uint32_t)(wi * (32 * 36 * 4));   // my warp's staging block
      if (wt < TM) sts32(s_nj + 4 * wt, __ldg(p.norms + row0 + j0 + wt));
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
      const float ni = __ldg(p.norms + row0 + i);
      float rs[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) rs[t] = 0.f;
      for (int cb = 0; cb < 2; ++cb) {
        // pass A (my row i, 32 columns): squared distances from the Gram into the staging block, and which of them the
        // Gram cannot be trusted for
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(64 * h + 32 * cb), v);
        const int jb = 64 * h + 32 * cb;
        unsigned flagged = 0u;
#pragma unroll
        for (int u = 0; u < 32; ++u) {
          const float nj = lds32(s_nj + 4 * (jb + u));
          const float d2 = fmaxf(ni + nj - 2.f * v[u], 0.f);
          // The 3xTF32 Gram leaves ~1e-6 (|xw_i|^2 + |xw_j|^2) of absolute error in d2.  It matters where it moves
          // W = exp(-d) (|dW| = W dd) or the metric gradient (~ W dd / d) by more than 1e-5: near-duplicates against the
          // (centred) norms (SURVEY Q7).  Far pairs (W ~ 0) never are.
          // Test: exp(-d) (ni + nj) > 20 min(d, d^2).  exp(-d) <= 1 settles almost every entry without sqrt / exp.
          const float sn = ni + nj;
          const bool maybe = d2 >= 1.f ? sn * sn > 400.f * d2 : sn > 20.f * d2;
          if (maybe && i != j0 + jb + u) {
            const float dg = sqrtf(d2);
            if (__expf(-dg) * sn > 20.f * fminf(dg, d2)) flagged |= 1u << u;
          }
          v[u] = d2;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
          sts128(stg + 4 * (lane * 36 + 4 * u), make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]));
        __syncwarp();
        // fix-up: flagged entries are recomputed from direct differences, the warp working together on one entry at a
        // time (lanes stride over the features), and patched in the staging block
        unsigned cols = __reduce_or_sync(0xffffffffu, flagged);
        while (cols) {
          const int u = __ffs(cols) - 1;
          cols &= cols - 1;
          const float* xj = p.XW + (row0 + j0 + jb + u) * (long long)F;
          unsigned todo = __ballot_sync(0xffffffffu, (flagged >> u) & 1u);
          while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const float* xs = p.XW + (row0 + m0 + q * 32 + src) * (long long)F;
            float acc = 0.f;
            for (int f = lane; f < F; f += 32) {
              const float df = __ldg(xs + f) - __ldg(xj + f);
              acc = fmaf(df, df, acc);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) sts32(stg + 4 * (src * 36 + u), acc);
          }
        }
        __syncwarp();
        // pass B, in the layout of the stores: lane holds row 4 t + lane / 8, columns 4 (lane & 7) ..
        const long long tile0 = (long long)g * n * n + (long long)(m0 + q * 32) * n + j0 + jb;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const int rr = 4 * t + (lane >> 3), c4 = 4 * (lane & 7);
          const float4 q2 = lds128(stg + 4 * (rr * 36 + c4));
          const int dj = (m0 + q * 32 + rr) - (j0 + jb + c4);   // the diagonal entry of this quad, if 0 <= dj < 4
          // sqrt as x rsqrt(x) and exp through ex2.approx: ~2 ulp each, far inside the 1e-4 of the parity tests, and a
          // third of the instructions of sqrtf / expf in a pass that is issue-bound
          auto root = [](float x) { return x > 0.f ? x * rsqrtf(x) : 0.f; };
          float4 d, w;
          d.x = dj == 0 ? 0.f : root(q2.x); w.x = dj == 0 ? 0.f : __expf(-d.x);
          d.y = dj == 1 ? 0.f : root(q2.y); w.y = dj == 1 ? 0.f : __expf(-d.y);
          d.z = dj == 2 ? 0.f : root(q2.z); w.z = dj == 2 ? 0.f : __expf(-d.z);
          d.w = dj == 3 ? 0.f : root(q2.w); w.w = dj == 3 ? 0.f : __expf(-d.w);
          rs[t] += (w.x + w.y) + (w.z + w.w);
          const long long o = tile0 + (long long)rr * n + c4;
          if (p.dist) *reinterpret_cast<float4*>(p.dist + o) = d;
          if (p.resW) *reinterpret_cast<float4*>(p.resW + o) = w;
        }
        __syncwarp();
      }
      if (p.rowpart) {
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          float r8 = rs[t];
          r8 += __shfl_xor_sync(0xffffffffu, r8, 1);
          r8 += __shfl_xor_sync(0xffffffffu, r8, 2);
          r8 += __shfl_xor_sync(0xffffffffu, r8, 4);
          if ((lane & 7) == 0) p.rowpart[(row0 + m0 + q * 32 + 4 * t + (lane >> 3)) * p.ncb + (j0 / 64 + h)] = r8;
        }
      }

    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;\n" ::"r"(tmem_base) : "memory");
}

// mu[g][f] = mean over the n rows of graph g (equal-size graphs: rows g n ..): grid (B, F / 32), block (32, 8)
__global__ void graph_mean_kernel(const float* __restrict__ X, int n, int F, float* __restrict__ mu) {
  __shared__ float red[8][33];
  const int g = blockIdx.x, f = blockIdx.y * 32 + threadIdx.x;
  float s = 0.f;
  if (f < F)
    for (int r = threadIdx.y; r < n; r += 8) s += X[((long long)g * n + r) * F + f];
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && f < F) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    mu[(long long)g * F + f] = t / (float)n;
  }
}

// |x_r - mu_g|^2 per packed row: one warp per row
__global__ void row_norms_kernel(const float* __restrict__ X, const float* __restrict__ mu, int n, long long R, int F,
                                 float* __restrict__ norms) {
  const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= R) return;
  const float* m = mu + (r / n) * F;
  float s = 0.f;
  for (int f = lane; f < F; f += 32) {
    const float v = X[r * F + f] - m[f];
    s = fmaf(v, v, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) norms[r] = s;
}

// ------------------------------------------------------------------------------------------------
// F <= 8: stream L once.  One CTA per 64-row tile, 8 warps.
// ------------------------------------------------------------------------------------------------
template <int FP>
__device__ __forceinline__ void thin_epilogue(const GroupedArgs& p, long long row, const float (&acc)[FP]) {
  const int F = p.F;
#pragma unroll
  for (int f = 0; f < FP; ++f) {
    if (f >= F) break;
    const long long o = row * F + f;
    float v = p.cmul * acc[f];
    if (p.add_identity) v = fmaf(p.cmul, p.In[o], v);
    if (p.Add) v += p.Add[o];
    if (p.Sub) v -= p.Sub[o];
    if (p.RowScale) v = fmaf(p.RowScale[row], p.ScaleIn[o], v);
    p.Out[o] = v;
    if (p.Out2) p.Out2[o] = v;
  }
}

// op = L: a warp owns 8 rows of the tile, four at a time; lanes stride over the columns (coalesced rows of L)
template <int FP>
__global__ void __launch_bounds__(256) grouped_thin_kernel(GroupedArgs p) {
  const int g = p.tile_graph[blockIdx.x], m0 = p.tile_row[blockIdx.x];
  const int n = p.n_nodes[g], F = p.F;
  const long long row0 = p.node_off[g];
  const float* __restrict__ Lg = p.L + p.lap_off[g];
  const float* __restrict__ In = p.In + row0 * F;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int pass = 0; pass < 2; ++pass) {
    const int i0 = m0 + warp * 8 + pass * 4;
    if (i0 >= n) break;
    float acc[4][FP];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int f = 0; f < FP; ++f) acc[r][f] = 0.f;
    const float* lrow[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) lrow[r] = Lg + (long long)min(i0 + r, n - 1) * n;  // rows past the end repeat the last one
#pragma unroll 2
    for (int j = lane; j < n; j += 32) {
      float l[4], x[FP];
#pragma unroll
      for (int r = 0; r < 4; ++r) l[r] = __ldg(lrow[r] + j);
#pragma unroll
      for (int f = 0; f < FP; ++f) x[f] = (f < F) ? __ldg(In + (long long)j * F + f) : 0.f;
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int f = 0; f < FP; ++f) acc[r][f] = fmaf(l[r], x[f], acc[r][f]);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int f = 0; f < FP; ++f)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[r][f] += __shfl_xor_sync(0xffffffffu, acc[r][f], o);
    if (lane < 4 && i0 + lane < n) {
      float mine[FP];
#pragma unroll
      for (int f = 0; f < FP; ++f) {
        mine[f] = acc[0][f];
#pragma unroll
        for (int r = 1; r < 4; ++r)
          if (lane == r) mine[f] = acc[r][f];
      }
      thin_epilogue<FP>(p, row0 + i0 + lane, mine);
    }
  }
}

// op = L^T: lane = output row of a 32-row segment (coalesced along the rows of L), the 8 warps are
// 2 segments x 4 interleaved quarters of the contraction, summed through shared memory
template <int FP>
__global__ void __launch_bounds__(256) grouped_thin_kernel_t(GroupedArgs p) {
  __shared__ float red[3][64][FP + 1];
  const int g = p.tile_graph[blockIdx.x], m0 = p.tile_row[blockIdx.x];
  const int n = p.n_nodes[g], F = p.F;
  const long long row0 = p.node_off[g];
  const float* __restrict__ Lg = p.L + p.lap_off[g];
  const float* __restrict__ In = p.In + row0 * F;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int seg = warp & 1, jq = warp >> 1;
  const int il = seg * 32 + lane, i = m0 + il;
  float acc[FP];
#pragma unroll
  for (int f = 0; f < FP; ++f) acc[f] = 0.f;
  if (i < n) {
#pragma unroll 4
    for (int j = jq; j < n; j += 4) {
      const float l = __ldg(Lg + (long long)j * n + i);
#pragma unroll
      for (int f = 0; f < FP; ++f)
        if (f < F) acc[f] = fmaf(l, __ldg(In + (long long)j * F + f), acc[f]);
    }
  }
  if (jq > 0) {
#pragma unroll
    for (int f = 0; f < FP; ++f) red[jq - 1][il][f] = acc[f];
  }
  __syncthreads();
  if (jq == 0 && i < n) {
#pragma unroll
    for (int f = 0; f < FP; ++f) acc[f] += red[0][il][f] + red[1][il][f] + red[2][il][f];
    thin_epilogue<FP>(p, row0 + i, acc);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

}  // namespace bt

bool grouped_tc_supported(const GroupedArgs& g) {
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (g.F < 16 || (g.F & 3)) return false;
  return al16(g.In) && al16(g.Out) && al16(g.Out2) && al16(g.Add) && al16(g.Sub) && al16(g.ScaleIn);
}

int grouped_tc(const agcn_plan* plan, int tiles, const GroupedArgs& g, cudaStream_t st) {
  using namespace bt;
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return AGCN_ERR_CUDA;
  }
  // In as a [R, F] row-major matrix, boxes of 32 nodes x 32 columns, 128B swizzle with 32B atoms (MN-major TF32 operand)
  CUtensorMap map;
  cuuint64_t gdim[2] = {(cuuint64_t)g.F, (cuuint64_t)plan->R};
  cuuint64_t gstride[1] = {(cuuint64_t)g.F * sizeof(float)};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(g.In), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (grouped_tc) failed with code " + std::to_string((int)r));
    return AGCN_ERR_CUDA;
  }
  dim3 grid(tiles, (g.F + BN - 1) / BN);
  // equal-size graphs with 128-row tiles that all exist and 16-byte aligned rows of L: TMA-staged L tiles, A in TMEM
  const int un = plan->uniform_n;
  // ... when there are more 128-row CTAs than SMs (two of them share an SM and hide each other's latencies; with at most
  // one per SM the deeper rings of grouped_tc_kernel win: N = 4096, B = 4 measured 0.91 against 0.70 ms per layer)
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (un > 0 && un % TM == 0 && (reinterpret_cast<uintptr_t>(g.L) & 15) == 0 && tiles == plan->large_tiles &&
      (long long)plan->B * un < (1ll << 31) && ((long long)(tiles / 2) * grid.y > sms || g.force_uniform)) {
    CUtensorMap mapL;
    cuuint64_t ld[2] = {(cuuint64_t)un, (cuuint64_t)plan->B * un};
    cuuint64_t ls[1] = {(cuuint64_t)un * sizeof(float)};
    cuuint32_t lbox[2] = {32, 128};
    if (g.transL) { lbox[0] = 128; lbox[1] = 32; }
    r = fn(&mapL, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(g.L), ld, ls, lbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
           g.transL ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("cuTensorMapEncodeTiled (grouped_tcu, L) failed with code " + std::to_string((int)r));
      return AGCN_ERR_CUDA;
    }
    static std::once_flag once_u;
    std::call_once(once_u, [] {
      cudaFuncSetAttribute(grouped_tcu_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, U_SMEM);
    });
    {
      ProfScope prof("bt::grouped_tcu_kernel", st);
      grouped_tcu_kernel<<<grid, U_THREADS, U_SMEM, st>>>(map, mapL, g, un);
    }
    AGCN_LAUNCH_CHECK();
    return AGCN_OK;
  }
  static std::once_flag once;
  std::call_once(once, [] {
    cudaFuncSetAttribute(grouped_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL);
  });
  {
    ProfScope prof("bt::grouped_tc_kernel", st);
    grouped_tc_kernel<<<grid, THREADS, SMEM_TOTAL, st>>>(map, g);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// ---- pair matrices of big equal-size graphs on the tensor cores (see pair_tcu_kernel)
bool pair_tc_supported(const agcn_plan* plan, int F) {
  const int un = plan->uniform_n;
  return un > 0 && un % bt::TM == 0 && F % bt::BK == 0 && F >= bt::BK && F <= 256 && plan->big_tiles == plan->large_tiles &&
         plan->big_tiles > 0 && (long long)plan->B * un * 8 < (1ll << 31);
}

static int pair_map(CUtensorMap* map, const float* ptr, uint64_t rows, int F) {
  using namespace bt;
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return AGCN_ERR_CUDA;
  }
  cuuint64_t gdim[2] = {(cuuint64_t)F, rows};
  cuuint64_t gstride[1] = {(cuuint64_t)F * sizeof(float)};
  cuuint32_t box[2] = {32, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (pair_tc) failed with code " + std::to_string((int)r));
    return AGCN_ERR_CUDA;
  }
  return AGCN_OK;
}

static int pair_launch(const agcn_plan* plan, const CUtensorMap& mA, const CUtensorMap& mB0, const CUtensorMap& mB1,
                       bt::PairTcArgs& k, const char* name, cudaStream_t st) {
  using namespace bt;
  k.tile_graph = plan->d_tile_graph; k.tile_row = plan->d_tile_row;
  k.n = plan->uniform_n; k.R = (int)plan->R;
  static std::once_flag once;
  constexpr int P_SMEM = U_SMEM + 1024;   // + the graph's mean row
  std::call_once(once, [] {
    cudaFuncSetAttribute(pair_tcu_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, U_SMEM + 1024);
    cudaFuncSetAttribute(pair_tcu_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, U_SMEM + 1024);
  });
  dim3 grid(plan->big_tiles, plan->uniform_n / TM);
  {
    ProfScope prof(name, st);
    if (k.mode)
      pair_tcu_kernel<true><<<grid, U_THREADS, P_SMEM, st>>>(mA, mB0, mB1, k);
    else
      pair_tcu_kernel<false><<<grid, U_THREADS, P_SMEM, st>>>(mA, mB0, mB1, k);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

// SIM: dist / resW / rowpart of every big graph from XW [R, F]; norms: scratch of R + 64 + B F floats
int pair_tc_similarity(const agcn_plan* plan, const float* XW, int F, float* norms, float* dist, float* resW, float* rowpart,
                       int ncb, cudaStream_t st) {
  using namespace bt;
  float* mu = norms + ((plan->R + 63) & ~(int64_t)63);   // scratch: norms [R] then mu [B][F]
  graph_mean_kernel<<<dim3(plan->B, (F + 31) / 32), dim3(32, 8), 0, st>>>(XW, plan->uniform_n, F, mu);
  AGCN_LAUNCH_CHECK();
  row_norms_kernel<<<(unsigned)((plan->R * 32 + 255) / 256), 256, 0, st>>>(XW, mu, plan->uniform_n, plan->R, F, norms);
  AGCN_LAUNCH_CHECK();
  CUtensorMap m;
  int rc;
  if ((rc = pair_map(&m, XW, (uint64_t)plan->R, F))) return rc;
  PairTcArgs k{};
  k.F = F; k.S = 1; k.mode = 0;
  k.XW = XW; k.mu = mu; k.norms = norms; k.dist = dist; k.resW = resW; k.rowpart = rowpart; k.ncb = ncb;
  return pair_launch(plan, m, m, m, k, "bt::pair_tcu_kernel<SIM>", st);
}

// DL: dL = dL_in + sum_{k=1}^{K-1} c_k U_k T_{k-1}^T; U = [K][R][F] (slice k = U_k), X = T_0, T = T_1 .. T_{K-1}
int pair_tc_dL(const agcn_plan* plan, const float* U, const float* X, const float* T, int F, int K, const float* dL_in,
               float* dL, cudaStream_t st) {
  using namespace bt;
  CUtensorMap mA, mB0, mB1;
  int rc;
  if ((rc = pair_map(&mA, U, (uint64_t)K * plan->R, F))) return rc;
  if ((rc = pair_map(&mB0, X, (uint64_t)plan->R, F))) return rc;
  if ((rc = pair_map(&mB1, K > 2 ? T : X, (uint64_t)(K > 2 ? (K - 2) : 1) * plan->R, F))) return rc;
  PairTcArgs k{};
  k.F = F; k.S = K - 1; k.mode = 1;
  k.dL_in = dL_in; k.out = dL;
  return pair_launch(plan, mA, mB0, mB1, k, "bt::pair_tcu_kernel<DL>", st);
}

bool grouped_thin_supported(const GroupedArgs& g) {
  return g.F >= 1 && g.F <= 8;
}

int grouped_thin(int tiles, const GroupedArgs& g, cudaStream_t st) {
  using namespace bt;
  if (g.F <= 4) {
    if (g.transL)
      {
        ProfScope prof("bt::grouped_thin_kernel", st);
        grouped_thin_kernel_t<4><<<tiles, 256, 0, st>>>(g);
      }
    else
      {
        ProfScope prof("bt::grouped_thin_kernel", st);
        grouped_thin_kernel<4><<<tiles, 256, 0, st>>>(g);
      }
  } else {
    if (g.transL)
      {
        ProfScope prof("bt::grouped_thin_kernel", st);
        grouped_thin_kernel_t<8><<<tiles, 256, 0, st>>>(g);
      }
    else
      {
        ProfScope prof("bt::grouped_thin_kernel", st);
        grouped_thin_kernel<8><<<tiles, 256, 0, st>>>(g);
      }
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // namespace agcn
