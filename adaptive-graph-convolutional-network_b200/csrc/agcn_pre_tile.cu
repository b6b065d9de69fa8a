// Transform product (the dense contraction of a layer) on the tensor cores.  GENERIC kernel first: 128-row ranges ("pre tiles") of
// graphs above AGCN_FUSE_MAX_N nodes -- the mid-size molecules of a Tox21 / ToxCast batch and every point cloud.  Their
// Chebyshev recurrences run in the per-graph / row-tiled kernels (agcn_graph_small.cu, agcn_big_tc.cu); what is left
// per 128-row range is a plain dense contraction on the tensor cores:
//
//   forward   Y = act(sum_s T_s W_s + b)        graphconv.py:238-247, :118-123   (T_0 = X, T_s saved by the recurrences)
//   backward  G_z = dYpre W_z^T, z = 0..K-1     dYpre = dY * relu'(Y); input of the reverse recurrences
//
// One CTA per range.  Every hand-off ("item") is one 32-column chunk of one operand matrix: the 8 worker warps
// (thread = tile row x column half) load their 16 values from global memory one item ahead, split them into hi / lo TF32
// halves and write them once into a K-major SWIZZLE_128B operand slot; TMA brings the matching pre-split parameter
// tile; one thread issues the 3xTF32 products into a TMEM accumulator.  Items are independent, so three slots keep
// loads, splits and tensor-core work of consecutive items in flight together (0.4 .. 0.5 us per item against 0.9 us
// + a dependent recurrence step in the fused tile kernel's hand-off; profiles/r02_b_tile_v2_timeline_ts_n64_staged.txt).
#include <cuda.h>

#include <algorithm>
#include <mutex>

#include "agcn_internal.cuh"

namespace agcn {
namespace pt {

constexpr int TM = 128;            // rows per tile (UMMA M)
constexpr int CH = 32;             // feature columns per chunk = 128 bytes = one swizzle row
constexpr int UMMA_K = 8;          // tf32
constexpr int A_BYTES = TM * CH * 4;   // 16 KB: one half (hi or lo) of a rows x chunk operand
constexpr int WORKERS = 256;       // warps 2..9: two threads per tile row (column halves)
constexpr int THREADS = 64 + WORKERS;
constexpr int SLOTS = 3;

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

// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row atoms of 1024 bytes
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
               : "memory");
}
// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float v[16]) {
  uint32_t u[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void sts128(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};\n" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ int ldsi32(uint32_t a) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];\n" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }

// My half (16 columns: 16-byte groups 4h .. 4h+3) of row `row` of a rows x chunk operand ([128][32] K-major,
// SWIZZLE_128B), split into hi / lo TF32 halves.
__device__ __forceinline__ void write_rows_operand(uint32_t a_hi, uint32_t a_lo, int row, int h, const float v[16]) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float4 hi, lo;
    hi.x = tf32_rn(v[4 * g]);     hi.y = tf32_rn(v[4 * g + 1]);
    hi.z = tf32_rn(v[4 * g + 2]); hi.w = tf32_rn(v[4 * g + 3]);
    lo.x = tf32_rn(v[4 * g] - hi.x);     lo.y = tf32_rn(v[4 * g + 1] - hi.y);
    lo.z = tf32_rn(v[4 * g + 2] - hi.z); lo.w = tf32_rn(v[4 * g + 3] - hi.w);
    const uint32_t off = (uint32_t)(row * 128 + (((4 * h + g) ^ (row & 7)) << 4));
    sts128(a_hi + off, hi);
    sts128(a_lo + off, lo);
  }
}

struct SmemPlan {
  int w_bytes;     // one half of a parameter tile: N x 128 bytes
  int slot_bytes;  // rows operand (hi, lo) + parameter tile (hi, lo)
  int off_bars;
  int total;
};
__host__ __device__ inline SmemPlan smem_plan(int N) {
  SmemPlan s;
  s.w_bytes = N * 128;
  s.slot_bytes = 2 * A_BYTES + 2 * s.w_bytes;
  s.off_bars = SLOTS * s.slot_bytes;
  s.total = s.off_bars + 256 + 1024;  // + alignment slack
  return s;
}

struct PreArgs {
  const int4* tile_graphs;     // 2 x int4 per entry: {g, row_start, nrows, -1}, {node_off, ...}; NULL: tile t = packed
  const int32_t* tile_gstart;  // [tiles + 1]                                            rows [128 t, 128 t + 128) of all R
  int tile0;                   // first tile of this launch
  int R;                       // packed rows (all-rows mode)
  int Fin;                     // columns of the operand matrices: F forward, Fo backward
  int Fout;                    // columns of the result: Fo forward, F backward
  int K;
  int N;                       // MMA N (Fout padded to 16)
  int nchunks;                 // ceil(Fin / 32)
  int tmem_cols;               // allocation: acc_stride (forward) or 2 * acc_stride (backward: two accumulators)
  int acc_stride;              // power of two >= N
  const float* In;             // [R, Fin]   forward: X, backward: dY
  const float* Mask;           // backward: Y (dYpre = dY * [Y > 0]) or NULL
  const float* T;              // forward: saved T_1 .. T_{K-1}, [K-1][R][Fin]
  long long t_slice;
  const float* bias;           // forward
  int act;
  float* Out;                  // forward: Y [R, Fout]; backward: G [K][R][Fout]
  long long out_slice;         // backward: elements between G_z
  int forward;
};

__global__ void __launch_bounds__(THREADS, 1)
pre_tile_kernel(const __grid_constant__ CUtensorMap tmBhi, const __grid_constant__ CUtensorMap tmBlo, PreArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(base);
  const SmemPlan sp = smem_plan(p.N);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + sp.off_bars);
  uint64_t* full_bar = bars;            // [SLOTS] parameter tile landed (TMA)
  uint64_t* ops_bar = bars + SLOTS;     // [SLOTS] operand rows written by the 8 worker warps
  uint64_t* done_bar = bars + 2 * SLOTS;  // [SLOTS] the MMAs that read the slot retired
  uint64_t* out_bar = bars + 3 * SLOTS;     // accumulator complete (forward: once; backward: once per z)
  uint64_t* outfree_bar = bars + 3 * SLOTS + 1;  // backward: accumulator drained by the workers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * SLOTS + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = p.tile0 + blockIdx.x;
  const int K = p.K, N = p.N, nc = p.nchunks, Fin = p.Fin, Fout = p.Fout;
  // forward: ONE accumulation over all (chunk, s) items; backward: K passes over the chunks, one G_z each
  const int passes = p.forward ? 1 : K;
  const int per_pass = p.forward ? nc * K : nc;

  if (threadIdx.x == 0) {
    for (int s = 0; s < SLOTS; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&ops_bar[s], WORKERS / 32);
      mbar_init(&done_bar[s], 1);
    }
    mbar_init(out_bar, 1);
    mbar_init(outfree_bar, WORKERS / 32);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    const uint32_t s = smem_u32(tmem_slot);
    switch (p.tmem_cols) {
      case 32: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 32;\n" ::"r"(s) : "memory"); break;
      case 64: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;\n" ::"r"(s) : "memory"); break;
      case 128: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;\n" ::"r"(s) : "memory"); break;
      default: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;\n" ::"r"(s) : "memory"); break;
    }
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // item t of a pass: forward (chunk, s) = (t / K, t % K); backward chunk t of pass z.  Parameter tile (chunk, slice).
  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int t_all = 0;
      for (int z = 0; z < passes; ++z)
        for (int t = 0; t < per_pass; ++t, ++t_all) {
          const int slot = t_all % SLOTS, u = t_all / SLOTS;
          if (u > 0) mbar_wait(&done_bar[slot], (uint32_t)((u - 1) & 1));
          const int cc = p.forward ? t / K : t, sl = p.forward ? t % K : z;
          const uint32_t dst = sbase + slot * sp.slot_bytes + 2 * A_BYTES;
          mbar_expect_tx(&full_bar[slot], 2 * sp.w_bytes);
          tma_load_2d(dst, &tmBhi, &full_bar[slot], cc * CH, sl * N);
          tma_load_2d(dst + sp.w_bytes, &tmBlo, &full_bar[slot], cc * CH, sl * N);
        }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      // D = f32, A = B = tf32, both K-major
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
      int t_all = 0;
      for (int z = 0; z < passes; ++z) {
        if (z > 1) {   // accumulator z & 1 was last used by pass z - 2: wait until the workers have drained it
          mbar_wait(outfree_bar, (uint32_t)((z - 2) & 1));
          tc_fence_after();
        }
        const uint32_t acc = tmem_base + (uint32_t)((z & 1) * p.acc_stride);
        for (int t = 0; t < per_pass; ++t, ++t_all) {
          const int slot = t_all % SLOTS, u = t_all / SLOTS;
          mbar_wait(&full_bar[slot], (uint32_t)(u & 1));
          mbar_wait(&ops_bar[slot], (uint32_t)(u & 1));
          tc_fence_after();
          const uint32_t sa = sbase + slot * sp.slot_bytes, sa_lo = sa + A_BYTES;
          const uint32_t sw = sa + 2 * A_BYTES, sw_lo = sw + sp.w_bytes;
#pragma unroll
          for (int k = 0; k < CH / UMMA_K; ++k) {
            const uint32_t koff = k * UMMA_K * 4;
            const uint64_t a_hi = make_desc(sa + koff), a_lo = make_desc(sa_lo + koff);
            const uint64_t b_hi = make_desc(sw + koff), b_lo = make_desc(sw_lo + koff);
            umma_ss(acc, a_lo, b_hi, idesc, (t | k) != 0);
            umma_ss(acc, a_hi, b_lo, idesc, 1);
            umma_ss(acc, a_hi, b_hi, idesc, 1);
          }
          umma_commit(&done_bar[slot]);
        }
        umma_commit(out_bar);
      }
    }
  } else {
    // ================= workers =================
    const int q = warp & 3;             // TMEM lane quarter of this warp
    const int h = (warp - 2) >> 2;      // column half
    const int r = q * 32 + lane;        // my tile row
    int grow = -1;
    if (p.tile_graphs) {
      const int4 e0 = __ldg(p.tile_graphs + 2 * p.tile_gstart[tile]);       // {g, row_start, nrows, -1}
      const int4 e1 = __ldg(p.tile_graphs + 2 * p.tile_gstart[tile] + 1);   // {node_off, ...}
      if (r < e0.z) grow = e1.x + e0.y + r;
    } else if (tile * TM + r < p.R) {
      grow = tile * TM + r;   // the contraction does not care about graph boundaries
    }
    const bool vecIn = ((Fin & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.In) & 15) == 0) &&
                       (!p.Mask || (reinterpret_cast<uintptr_t>(p.Mask) & 15) == 0) &&
                       (!p.T || (((reinterpret_cast<uintptr_t>(p.T) & 15) == 0) && ((p.t_slice & 3) == 0)));
    // my 16 columns of chunk cc of operand matrix sl (forward: T_sl; backward: dY with Y for the relu' mask), as RAW
    // values: the mask is applied when the item is consumed -- a compare at load time would wait for the load and
    // turn the prefetch into a stall (ncu source view of the first version: all top stalls on those FSETPs)
    auto load_item = [&](int cc, int sl, float v[16], float m[16]) {
      const int c0 = cc * CH + 16 * h;
      const float* src = (p.forward && sl > 0) ? p.T + (long long)(sl - 1) * p.t_slice : p.In;
      const float* msk = p.forward ? nullptr : p.Mask;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int col = c0 + 4 * g;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f), y = make_float4(1.f, 1.f, 1.f, 1.f);
        if (grow >= 0 && col < Fin) {
          const long long o = (long long)grow * Fin + col;
          if (vecIn) {
            x = __ldg(reinterpret_cast<const float4*>(src + o));
            if (msk) y = __ldg(reinterpret_cast<const float4*>(msk + o));
          } else {
            float t[4] = {0.f, 0.f, 0.f, 0.f}, ty[4] = {1.f, 1.f, 1.f, 1.f};
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (col + e < Fin) {
                t[e] = __ldg(src + o + e);
                if (msk) ty[e] = __ldg(msk + o + e);
              }
            x = make_float4(t[0], t[1], t[2], t[3]);
            y = make_float4(ty[0], ty[1], ty[2], ty[3]);
          }
        }
        v[4 * g] = x.x; v[4 * g + 1] = x.y; v[4 * g + 2] = x.z; v[4 * g + 3] = x.w;
        m[4 * g] = y.x; m[4 * g + 1] = y.y; m[4 * g + 2] = y.z; m[4 * g + 3] = y.w;
      }
    };
    auto coords = [&](int z, int t, int& cc, int& sl) {
      cc = p.forward ? t / K : t;
      sl = p.forward ? t % K : z;
    };
    // accumulator -> global rows (bias + activation in the forward direction)
    auto drain_out = [&](float* dstm, uint32_t acc_col) {
      const bool vecO = ((Fout & 3) == 0) && ((reinterpret_cast<uintptr_t>(dstm) & 15) == 0);
      for (int c0 = 16 * h; c0 < N && c0 < Fout; c0 += 32) {
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + acc_col + (uint32_t)c0, v);
        if (grow < 0) continue;
        if (p.forward) {
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            float o = v[u] + ((p.bias && c0 + u < Fout) ? __ldg(p.bias + c0 + u) : 0.f);
            if (p.act == AGCN_ACT_RELU) o = fmaxf(o, 0.f);
            v[u] = o;
          }
        }
        float* dst = dstm + (long long)grow * Fout + c0;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (c0 + 4 * g >= Fout) continue;
          if (vecO && c0 + 4 * g + 3 < Fout) {
            *reinterpret_cast<float4*>(dst + 4 * g) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (c0 + 4 * g + e < Fout) dst[4 * g + e] = v[4 * g + e];
          }
        }
      }
    };

    // Items are independent: the values of item t + 2 are requested before item t is split and handed over (two pairs
    // of register buffers, the loop unrolled by two so that they stay registers).
    const int total = passes * per_pass;
    auto fetch = [&](int idx, float (&buf)[16], float (&mk)[16]) {
      if (idx >= total) return;
      const int z = idx / per_pass, t = idx - z * per_pass;
      int cc, sl;
      coords(z, t, cc, sl);
      load_item(cc, sl, buf, mk);
    };
    auto process = [&](int idx, float (&buf)[16], float (&mk)[16]) {
      if (idx >= total) return;
      float v[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] = (mk[e] > 0.f) ? buf[e] : 0.f;   // relu'(0) = 0 (TF's ReluGrad); forward: mk = 1
      fetch(idx + 2, buf, mk);
      const int slot = idx % SLOTS, u = idx / SLOTS;
      if (u > 0) {
        if (lane == 0) mbar_wait(&done_bar[slot], (uint32_t)((u - 1) & 1));
        __syncwarp();
      }
      const uint32_t st = sbase + slot * sp.slot_bytes;
      write_rows_operand(st, st + A_BYTES, r, h, v);
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) mbar_arrive(&ops_bar[slot]);
      const int z = idx / per_pass;
      if (idx - z * per_pass == per_pass - 1) {
        // last item of pass z handed over: drain pass z - 1 (its MMAs finished long ago; pass z's are still running
        // on the other accumulator), and the last pass itself at the very end
        for (int zd = (z > 0 ? z - 1 : z); zd <= z; ++zd) {
          if (zd == z && z != passes - 1) break;
          if (lane == 0) mbar_wait(out_bar, (uint32_t)(zd & 1));
          __syncwarp();
          tc_fence_after();
          drain_out(p.forward ? p.Out : p.Out + (long long)zd * p.out_slice, (uint32_t)((zd & 1) * p.acc_stride));
          tc_fence_before();
          __syncwarp();
          if (lane == 0 && zd + 2 < passes) mbar_arrive(outfree_bar);   // only pass zd + 2 waits for this accumulator
        }
      }
    };
    float b0[16], m0[16], b1[16], m1[16];
    fetch(0, b0, m0);
    fetch(1, b1, m1);
    for (int idx = 0; idx < total; idx += 2) {
      process(idx, b0, m0);
      process(idx + 1, b1, m1);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    switch (p.tmem_cols) {
      case 32: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 32;\n" ::"r"(tmem_base) : "memory"); break;
      case 64: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;\n" ::"r"(tmem_base) : "memory"); break;
      case 128: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;\n" ::"r"(tmem_base) : "memory"); break;
      default: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;\n" ::"r"(tmem_base) : "memory"); break;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Contraction over ALL packed rows (the layer's main product since the recurrences moved to agcn_cheb_tile.cu):
//
//   forward   Y[r, :]   = act(sum_s T_s[r, :] W_s + b)          one accumulator, items (chunk, s), one W tile per item
//   backward  G_z[r, :] = (dY * relu'(Y))[r, :] W_z^T, z < K    K accumulators, items = chunks of dYpre, K W tiles per item
//
// What the generic kernel above (and the fused tile kernels before it) got wrong, from ncu + SASS (profiles/r02h_*):
//  * `fence.proxy.async` -- required between the workers' generic-proxy writes of an operand slot and the tensor core's
//    reads -- is lowered to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC: the MEMBAR waits for every global load the thread has in
//    flight, so register prefetch of the next items never overlapped anything and every item paid a full L2 / HBM round
//    trip (~1.5 us per item against 0.4 us of tensor-core work);
//  * ~450 instructions per thread and item of address arithmetic, bounds predicates and integer divisions;
//  * the backward direction loaded and split the same dYpre chunk once per z.
// Here NO thread that fences ever issues a global load: one producer thread streams the raw fp32 row tiles (128 rows x
// 32 columns, SWIZZLE_128B) into a staging ring with TMA, a second one the pre-split parameter tiles; the 8 worker warps
// read a staged tile from shared memory, split it into hi / lo TF32 halves (relu' mask applied from the staged Y tile in
// the backward direction) and write them into an operand slot in TENSOR MEMORY (tcgen05.st; the MMAs take A from TMEM):
//  * a tf32 MMA with both operands in shared memory reads 8 KB per 64 cycles at N = 128 -- all of the SM's 128 B/clk --
//    so the workers' own loads / stores and the TMA writes of the next tiles fought the tensor core for the same port
//    (per-CTA globaltimer timeline: 1.0 us to split and store one 16 KB item, 1.4 us per item against 0.4 us of MMA work);
//  * with A in tensor memory the MMAs read only the parameter tile (64 B/clk) and the workers never write shared memory,
//    so no proxy fence at all.
// Every dYpre chunk is split ONCE and multiplied with its K parameter tiles.  Requires Fin % 32 == 0, 16-byte aligned
// rows and accumulators + one operand slot within the 512 TMEM columns (else the generic kernel).
// Rings: NS staged raw tiles (16 KB, backward 2 x 16 KB), NA operand slots in TMEM (hi | lo, 64 columns), NB parameter
// tiles (hi | lo, 2 x N x 128 bytes).
// ------------------------------------------------------------------------------------------------
constexpr int RG_THREADS = 96 + WORKERS;   // warp 0: parameter tiles, warp 1: MMA, warp 2: raw row tiles, warps 3..10 workers

struct RowsArgs {
  int R, Fin, Fout, K, N, nchunks;
  int NS, NA, NB;              // ring depths
  int acc_stride, tmem_cols;
  int full_tiles;              // backward: CTAs [0, full_tiles) own a whole tile (all K accumulators); the tiles behind them
                               // (the partial last wave) are split over K CTAs, one G_z each
  int a_col0;                  // first TMEM column of the operand slots (behind the accumulators): slot s = [hi 32 | lo 32]
  int has_mask;                // backward: the second staged tile is Y (relu' mask)
  const float* bias;
  int act;
  float* Out;                  // forward: Y; backward: G [K][R][Fout]
  long long out_slice;
};

// D[tmem] (+)= A[tmem] * B[smem]   (A: lane = row, one 32-bit column per K element)
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// 16 consecutive columns of this thread's TMEM lane <- registers
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float v[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }

__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];\n" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}

template <bool FWD>
__global__ void __launch_bounds__(RG_THREADS, FWD ? 2 : 1)
rows_gemm_kernel(const __grid_constant__ CUtensorMap tmBhi, const __grid_constant__ CUtensorMap tmBlo,
                 const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmAux, RowsArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = smem_u32(base);
  const int NS = p.NS, NA = p.NA, NB = p.NB, N = p.N, K = p.K, nc = p.nchunks;
  const int w_bytes = N * 128;
  const int stage_bytes = (!FWD && p.has_mask) ? 2 * A_BYTES : A_BYTES;
  const uint32_t b_ring = sbase, s_ring = b_ring + (uint32_t)(NB * 2 * w_bytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + NB * 2 * w_bytes + NS * stage_bytes);
  uint64_t* a_full = bars;          // [NA] operand rows written to tensor memory by the 8 worker warps
  uint64_t* a_empty = bars + 4;     // [NA] the MMAs that read the slot retired
  uint64_t* b_full = bars + 8;      // [NB] parameter tile landed (TMA)
  uint64_t* b_empty = bars + 12;    // [NB] the MMAs that read the tile retired
  uint64_t* s_full = bars + 16;     // [NS] raw row tile landed (TMA)
  uint64_t* s_empty = bars + 20;    // [NS] the 8 worker warps have read it
  uint64_t* out_bar = bars + 24;    // every accumulator complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 25);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // backward, partial last wave: tile full_tiles + e / K, accumulator z0 = e % K only
  const bool split = !FWD && (int)blockIdx.x >= p.full_tiles;
  const int tile = split ? p.full_tiles + ((int)blockIdx.x - p.full_tiles) / K : (int)blockIdx.x;
  const int z0 = split ? ((int)blockIdx.x - p.full_tiles) % K : 0;
  const int items = FWD ? nc * K : nc;          // row-operand items
  const int nb = FWD ? 1 : (split ? 1 : K);     // parameter tiles per item

  if (threadIdx.x == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(&a_full[s], WORKERS / 32);
      mbar_init(&a_empty[s], 1);
      mbar_init(&b_full[s], 1);
      mbar_init(&b_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&s_empty[s], WORKERS / 32);
    }
    mbar_init(out_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    const uint32_t s = smem_u32(tmem_slot);
    switch (p.tmem_cols) {
      case 32: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 32;\n" ::"r"(s) : "memory"); break;
      case 64: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;\n" ::"r"(s) : "memory"); break;
      case 128: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;\n" ::"r"(s) : "memory"); break;
      case 256: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;\n" ::"r"(s) : "memory"); break;
      default: asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(s) : "memory"); break;
    }
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer of the parameter tiles =================
    if (lane == 0) {
      int bi = 0, cc = 0, sl = 0;
      for (int i = 0; i < items; ++i) {
        for (int j = 0; j < nb; ++j, ++bi) {
          const int slot = bi % NB, u = bi / NB;
          if (u > 0) mbar_wait(&b_empty[slot], (uint32_t)((u - 1) & 1));
          const uint32_t dst = b_ring + (uint32_t)(slot * 2 * w_bytes);
          const int z = FWD ? sl : z0 + j;
          mbar_expect_tx(&b_full[slot], 2 * w_bytes);
          tma_load_2d(dst, &tmBhi, &b_full[slot], cc * CH, z * N);
          tma_load_2d(dst + w_bytes, &tmBlo, &b_full[slot], cc * CH, z * N);
        }
        if (FWD) {
          if (++sl == K) { sl = 0; ++cc; }
        } else {
          ++cc;
        }
      }
    }
  } else if (warp == 2) {
    // ================= TMA producer of the raw row tiles =================
    if (lane == 0) {
      int cc = 0, sl = 0;
      for (int i = 0; i < items; ++i) {
        const int slot = i % NS, u = i / NS;
        if (u > 0) mbar_wait(&s_empty[slot], (uint32_t)((u - 1) & 1));
        const uint32_t dst = s_ring + (uint32_t)(slot * stage_bytes);
        mbar_expect_tx(&s_full[slot], stage_bytes);
        if (FWD) {
          if (sl == 0)
            tma_load_2d(dst, &tmIn, &s_full[slot], cc * CH, tile * TM);
          else   // T_sl: rows (sl - 1) * R + ... of the [(K-1) R, F] view of the saved terms
            tma_load_2d(dst, &tmAux, &s_full[slot], cc * CH, (sl - 1) * p.R + tile * TM);
          if (++sl == K) { sl = 0; ++cc; }
        } else {
          tma_load_2d(dst, &tmIn, &s_full[slot], cc * CH, tile * TM);
          if (p.has_mask) tma_load_2d(dst + A_BYTES, &tmAux, &s_full[slot], cc * CH, tile * TM);
          ++cc;
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
      int bi = 0;
      for (int i = 0; i < items; ++i) {
        const int aslot = i % NA;
        mbar_wait(&a_full[aslot], (uint32_t)((i / NA) & 1));
        tc_fence_after();
        const uint32_t ta_hi = tmem_base + (uint32_t)(p.a_col0 + aslot * 2 * CH), ta_lo = ta_hi + CH;
        for (int j = 0; j < nb; ++j, ++bi) {
          const int slot = bi % NB;
          mbar_wait(&b_full[slot], (uint32_t)((bi / NB) & 1));
          tc_fence_after();
          const uint32_t sw = b_ring + (uint32_t)(slot * 2 * w_bytes), sw_lo = sw + w_bytes;
          const uint32_t acc = tmem_base + (uint32_t)(FWD ? 0 : (z0 + j) * p.acc_stride);
#pragma unroll
          for (int k = 0; k < CH / UMMA_K; ++k) {
            const uint32_t koff = k * UMMA_K * 4;
            const uint64_t b_hi = make_desc(sw + koff), b_lo = make_desc(sw_lo + koff);
            umma_ts(acc, ta_lo + k * UMMA_K, b_hi, idesc, (i | k) != 0);
            umma_ts(acc, ta_hi + k * UMMA_K, b_lo, idesc, 1);
            umma_ts(acc, ta_hi + k * UMMA_K, b_hi, idesc, 1);
          }
          umma_commit(&b_empty[slot]);
        }
        umma_commit(&a_empty[aslot]);
      }
      umma_commit(out_bar);
    }
  } else {
    // ================= workers: staged raw tile -> hi / lo operand slot =================
    const int wi = warp - 3, q = warp & 3, h = wi >> 2, r = q * 32 + lane;
    const long long grow = (long long)tile * TM + r;
    const bool valid = grow < p.R;
    uint32_t soff[4];   // my four 16-byte groups of row r in a [128][32] SWIZZLE_128B tile (staged and operand alike)
#pragma unroll
    for (int g = 0; g < 4; ++g) soff[g] = (uint32_t)(r * 128 + (((4 * h + g) ^ (r & 7)) << 4));
    const bool masked = !FWD && p.has_mask;
    for (int i = 0; i < items; ++i) {
      const int sslot = i % NS, aslot = i % NA;
      if (lane == 0) {
        mbar_wait(&s_full[sslot], (uint32_t)((i / NS) & 1));
        if (i >= NA) mbar_wait(&a_empty[aslot], (uint32_t)((i / NA - 1) & 1));
      }
      __syncwarp();
      const uint32_t st = s_ring + (uint32_t)(sslot * stage_bytes);
      float4 x[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) x[g] = lds128(st + soff[g]);
      if (masked) {   // relu'(0) = 0 (TF's ReluGrad)
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 m = lds128(st + A_BYTES + soff[g]);
          x[g].x = m.x > 0.f ? x[g].x : 0.f; x[g].y = m.y > 0.f ? x[g].y : 0.f;
          x[g].z = m.z > 0.f ? x[g].z : 0.f; x[g].w = m.w > 0.f ? x[g].w : 0.f;
        }
      }
      // hi / lo TF32 halves of my 16 values -> my lane of the operand slot in tensor memory (columns 16h .. 16h+15)
      float hi[16], lo[16];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        hi[4 * g] = tf32_rn(x[g].x); hi[4 * g + 1] = tf32_rn(x[g].y);
        hi[4 * g + 2] = tf32_rn(x[g].z); hi[4 * g + 3] = tf32_rn(x[g].w);
        lo[4 * g] = tf32_rn(x[g].x - hi[4 * g]); lo[4 * g + 1] = tf32_rn(x[g].y - hi[4 * g + 1]);
        lo[4 * g + 2] = tf32_rn(x[g].z - hi[4 * g + 2]); lo[4 * g + 3] = tf32_rn(x[g].w - hi[4 * g + 3]);
      }
      const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(p.a_col0 + aslot * 2 * CH + 16 * h);
      tmem_st16(ta, hi);
      tmem_st16(ta + CH, lo);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&s_empty[sslot]);   // the staged tile is consumed (its values are in registers / tensor memory)
        mbar_arrive(&a_full[aslot]);
      }
    }
    // ---- drain
    if (lane == 0) mbar_wait(out_bar, 0);
    __syncwarp();
    tc_fence_after();
    const int Fout = p.Fout;
    const int zbeg = FWD ? 0 : z0, zend = FWD ? 1 : (split ? z0 + 1 : K);
    for (int z = zbeg; z < zend; ++z) {
      float* dstm = p.Out + (long long)z * p.out_slice;
      const bool vecO = ((Fout & 3) == 0) && ((reinterpret_cast<uintptr_t>(dstm) & 15) == 0);
      for (int c0 = 16 * h; c0 < N && c0 < Fout; c0 += 32) {
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(z * p.acc_stride + c0), v);
        if (!valid) continue;
        if (FWD) {
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            float o = v[u] + ((p.bias && c0 + u < Fout) ? __ldg(p.bias + c0 + u) : 0.f);
            if (p.act == AGCN_ACT_RELU) o = fmaxf(o, 0.f);
            v[u] = o;
          }
        }
        float* dst = dstm + grow * Fout + c0;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (c0 + 4 * g >= Fout) continue;
          if (vecO && c0 + 4 * g + 3 < Fout) {
            *reinterpret_cast<float4*>(dst + 4 * g) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (c0 + 4 * g + e < Fout) dst[4 * g + e] = v[4 * g + e];
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    switch (p.tmem_cols) {
      case 32: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 32;\n" ::"r"(tmem_base) : "memory"); break;
      case 64: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;\n" ::"r"(tmem_base) : "memory"); break;
      case 128: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;\n" ::"r"(tmem_base) : "memory"); break;
      case 256: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;\n" ::"r"(tmem_base) : "memory"); break;
      default: asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tmem_base) : "memory"); break;
    }
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

// [rows, cols] fp32 row-major, box = 32 columns x box_rows, 128-byte swizzle
static int make_map(CUtensorMap* map, const float* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return AGCN_ERR_CUDA;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)CH, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
    return AGCN_ERR_CUDA;
  }
  return AGCN_OK;
}


static int pad16(int x) { return (x + 15) & ~15; }
static int pad32(int x) { return (x + 31) & ~31; }

// fast path of the all-rows contraction: full 32-column chunks, 16-byte aligned rows, accumulators within TMEM
static bool rows_fast(const PreArgs& a) {
  auto al = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (a.Fin % CH != 0 || !al(a.In) || (a.Mask && !al(a.Mask)) || (a.T && (!al(a.T) || (a.t_slice & 3)))) return false;
  const int stride = a.N <= 32 ? 32 : (a.N <= 64 ? 64 : 128);
  return a.N <= 128 && (a.forward ? stride : a.K * stride) + 2 * CH <= 512;   // accumulators + one operand slot in TMEM
}

static int launch_rows(const agcn_plan* plan, const PreArgs& a, const CUtensorMap& mhi, const CUtensorMap& mlo, const char* name,
                       cudaStream_t st) {
  RowsArgs r{};
  r.R = (int)plan->R; r.Fin = a.Fin; r.Fout = a.Fout; r.K = a.K; r.N = a.N; r.nchunks = a.Fin / CH;
  r.acc_stride = a.N <= 32 ? 32 : (a.N <= 64 ? 64 : 128);
  r.a_col0 = a.forward ? r.acc_stride : a.K * r.acc_stride;
  // forward: two CTAs per SM (256 TMEM columns and ~100 KB of shared memory each): a batch of 155 row tiles is ONE
  // wave on 148 SMs instead of two, and two tiles on an SM hide each other's latencies
  const int tmem_budget = a.forward ? 256 : 512;
  r.NA = std::max(1, std::min(3, (tmem_budget - r.a_col0) / (2 * CH)));
  int cols = r.a_col0 + r.NA * 2 * CH, tm = 32;
  while (tm < cols) tm <<= 1;
  r.tmem_cols = tm;
  r.has_mask = (!a.forward && a.Mask) ? 1 : 0;
  r.bias = a.bias; r.act = a.act; r.Out = a.Out; r.out_slice = a.out_slice;
  // raw row tiles: [R, Fin] views of the operand matrices, box = 32 columns x 128 rows (rows beyond the tensor: zeros)
  CUtensorMap min, maux;
  int rc;
  if ((rc = make_map(&min, a.In, (uint64_t)plan->R, (uint64_t)a.Fin, (uint32_t)TM))) return rc;
  if (a.forward) {
    const float* aux = (a.K > 1) ? a.T : a.In;
    const uint64_t rows = (a.K > 1) ? (uint64_t)(a.K - 1) * plan->R : (uint64_t)plan->R;
    if ((rc = make_map(&maux, aux, rows, (uint64_t)a.Fin, (uint32_t)TM))) return rc;
  } else {
    if ((rc = make_map(&maux, a.Mask ? a.Mask : a.In, (uint64_t)plan->R, (uint64_t)a.Fin, (uint32_t)TM))) return rc;
  }
  // rings: staged raw tiles ~64 KB, the rest parameter tiles (at most 4); the operand slots live in tensor memory
  const int w2 = 2 * a.N * 128, budget = (a.forward ? 112 : 227) * 1024 - 1024 - 256;
  const int stage_bytes = r.has_mask ? 2 * A_BYTES : A_BYTES;
  r.NS = a.forward ? 2 : std::min(4, 65536 / stage_bytes);
  r.NB = std::max(1, std::min(4, (budget - r.NS * stage_bytes) / w2));
  const int smem = r.NB * w2 + r.NS * stage_bytes + 256 + 1024;
  int ntiles = (int)((plan->R + TM - 1) / TM);
  r.full_tiles = ntiles;
  if (!a.forward && a.K > 1) {
    // one CTA per SM: the tiles of a partial last wave are split over K CTAs (one accumulator each, a third of the work)
    int sms = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int rem = ntiles % sms;
    if (ntiles > sms && rem > 0 && rem * a.K <= sms) {
      r.full_tiles = ntiles - rem;
      ntiles = r.full_tiles + rem * a.K;
    }
  }
  static std::once_flag once;
  std::call_once(once, [] {
    cudaFuncSetAttribute(rows_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(rows_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  });
  {
    ProfScope prof(name, st);
    if (a.forward)
      rows_gemm_kernel<true><<<ntiles, RG_THREADS, smem, st>>>(mhi, mlo, min, maux, r);
    else
      rows_gemm_kernel<false><<<ntiles, RG_THREADS, smem, st>>>(mhi, mlo, min, maux, r);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

static int launch(const agcn_plan* plan, int tile0, int ntiles, PreArgs& a, const float* wsplit, int Kp, const char* name,
                  cudaStream_t st) {
  const long long half = (long long)a.K * a.N * Kp;
  CUtensorMap mhi, mlo;
  int rc;
  if ((rc = make_map(&mhi, wsplit, (uint64_t)a.K * a.N, (uint64_t)Kp, (uint32_t)a.N))) return rc;
  if ((rc = make_map(&mlo, wsplit + half, (uint64_t)a.K * a.N, (uint64_t)Kp, (uint32_t)a.N))) return rc;
  if (tile0 < 0 && rows_fast(a)) return launch_rows(plan, a, mhi, mlo, a.forward ? "pt::rows_gemm_kernel(fwd)" : "pt::rows_gemm_kernel(bwd)", st);
  if (tile0 >= 0) {
    a.tile_graphs = reinterpret_cast<const int4*>(plan->d_ft_entries);
    a.tile_gstart = plan->d_ft_gstart;
    a.tile0 = tile0;
  } else {   // every packed row, 128 at a time
    a.tile_graphs = nullptr;
    a.tile_gstart = nullptr;
    a.tile0 = 0;
    a.R = (int)plan->R;
    ntiles = (int)((plan->R + TM - 1) / TM);
  }
  a.nchunks = Kp / CH;
  a.acc_stride = a.N <= 32 ? 32 : (a.N <= 64 ? 64 : 128);
  a.tmem_cols = a.forward ? a.acc_stride : 2 * a.acc_stride;
  const SmemPlan sp = smem_plan(a.N);
  static std::once_flag once;
  std::call_once(once, [] {
    cudaFuncSetAttribute(pre_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  });
  {
    ProfScope prof(name, st);
    pre_tile_kernel<<<ntiles, THREADS, sp.total, st>>>(mhi, mlo, a);
  }
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // namespace pt

// Y = act(sum_s T_s W_s + b) over the 128-row ranges [tile0, tile0 + ntiles) of the plan's tile list, or (tile0 < 0) over
// every packed row; wsplit = the pre-split W_s of fused_fwd_prep
int pre_forward(const agcn_plan* plan, int tile0, int ntiles, const float* X, const float* T, const float* wsplit,
                const float* bias, int act, int F, int Fo, int K, float* Y, cudaStream_t st) {
  if (ntiles <= 0 && tile0 >= 0) return AGCN_OK;
  pt::PreArgs a{};
  a.Fin = F; a.Fout = Fo; a.K = K; a.N = pt::pad16(Fo);
  a.In = X; a.Mask = nullptr; a.T = T; a.t_slice = (long long)plan->R * F;
  a.bias = bias; a.act = act; a.Out = Y; a.out_slice = 0; a.forward = 1;
  return pt::launch(plan, tile0, ntiles, a, wsplit, pt::pad32(F), "pt::pre_tile_kernel(fwd)", st);
}

// G_z = dYpre W_z^T (z = 0..K-1) over the same ranges; wsplit = the pre-split W_z^T of fused_bwd_prep
int pre_backward(const agcn_plan* plan, int tile0, int ntiles, const float* dY, const float* Y, const float* wsplit, int F,
                 int Fo, int K, float* G, cudaStream_t st) {
  if (ntiles <= 0 && tile0 >= 0) return AGCN_OK;
  pt::PreArgs a{};
  a.Fin = Fo; a.Fout = F; a.K = K; a.N = pt::pad16(F);
  a.In = dY; a.Mask = Y; a.T = nullptr; a.t_slice = 0;
  a.bias = nullptr; a.act = AGCN_ACT_LINEAR; a.Out = G; a.out_slice = (long long)plan->R * F; a.forward = 0;
  return pt::launch(plan, tile0, ntiles, a, wsplit, pt::pad32(Fo), "pt::pre_tile_kernel(bwd)", st);
}

}  // namespace agcn
