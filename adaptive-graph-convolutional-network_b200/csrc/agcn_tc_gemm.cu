// Node-level GEMMs on the 5th-generation tensor cores (tcgen05), fp32 in / fp32 out with 3xTF32
// split-precision accumulation in TMEM.
//
//   C_z[M,N] (+)= act( sum_{s<S} A_s[M,Kd] * B_{z,s}[N,Kd]^T + bias )
//
// A_s are row-major node matrices (K-major operands, streamed by TMA with 128-byte swizzle);
// B is a small parameter matrix that a prep kernel rearranges to [N,Kd] K-major and splits into
// hi/lo TF32 halves once per call.  Every A tile is split in shared memory by four warps:
//   x = hi + lo,  hi = x with the 13 low mantissa bits cleared (exact in TF32),  lo = x - hi
//   D += A_lo B_hi + A_hi B_lo + A_hi B_hi        (error ~2^-21 relative: inside the 1e-4 budget,
//                                                  a single TF32 pass, ~5e-4, is not; SURVEY Q7 / H1)
// One CTA per 128-row tile: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM owner), warps 2-5 =
// operand splitter, then epilogue (TMEM -> registers -> global, bias + activation fused).
//
// Used for Y = act(sum_k T_k W_k + b) (graphconv.py:238-247), G_k = dY W_k^T, XW = X M_L
// (graphconv.py:164) and dX += dXW M_L^T.
#include <cuda.h>

#include <algorithm>
#include <mutex>

#include "agcn_internal.cuh"

namespace agcn {

namespace tc {

constexpr int BM = 128;      // rows per CTA tile (UMMA M)
constexpr int BK = 32;       // fp32 elements per k-block = 128 bytes = one swizzle row
constexpr int UMMA_K = 8;    // tf32
constexpr int A_TILE_BYTES = BM * BK * 4;  // 16 KB

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
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row atoms of 1024 bytes
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);  // start address, 16-byte units
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused with swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                    // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
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

struct Args {
  int M, N, Kd, S;
  int kb_per_slice;   // ceil(Kd / 32)
  int ksplit;         // split-K: grid.y = Z * ksplit, split ks handles k-blocks [ks * kb_per_split, ...) and writes
  int kb_per_split;   // its raw partial sums to C + (z * ksplit + ks) * sliceC (the host reduces them)
  int rows_slice1;    // row offset between A1 slices in the stacked 2-D view
  int b_rows_slice;   // rows of one B slice in the stacked [Z*S*Npad, Kd] view (= Npad)
  float* C;
  int ldc;
  long long sliceC;
  const float* bias;
  const float* scale;  // optional device scalar multiplying the product
  int act, accumulate;
  // fused weighted sigmoid cross-entropy epilogue (multitask head): C receives d loss / d logits
  const float* bce_y;
  const float* bce_w;
  int bce_ld;        // row pitch of bce_y / bce_w
  float bce_scale;
  float* loss_part;  // [CTAs][4]
};

// ST = 0: as many stages as one CTA per SM affords; ST = 2: two stages, so that TWO CTAs share an SM (wide, short
// contractions with fewer 128-column tiles than SMs: the multitask logits)
template <int BN, int ST = 0>
struct Smem {
  static constexpr int B_TILE_BYTES = BN * BK * 4;
  static constexpr int STAGE_BYTES = 2 * A_TILE_BYTES + 2 * B_TILE_BYTES;
  static constexpr int STAGES = ST > 0 ? ST : ((BN <= 64) ? 4 : 3);
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
};

// PROB: the multitask head's prediction epilogue (agcn_head_predict): C receives the two-class softmax of every column
// pair (2t, 2t+1) instead of the product, and with bce_y set the same pass adds up the weighted sigmoid cross-entropy
// exactly as the training epilogue does.  A lane owns 4 consecutive columns starting at a multiple of 4, so a pair never
// straddles lanes or tiles.
// L2: the regression head's weighted L2 takes the place of the sigmoid cross-entropy (DeepChem's
// MultitaskGraphRegressor, final_loss='weighted_L2': the loss term is (w (x - y))^2, C receives 2 w^2 (x - y) bce_scale).
// With PROB as well it is the regression head's prediction epilogue: C receives x itself, and with bce_y set the same
// loss terms are added up in the order of the training epilogue.
template <int BN, int ST = 0, bool PROB = false, bool L2 = false>
__global__ void __launch_bounds__(192, ST == 2 ? 2 : 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmBhi, const __grid_constant__ CUtensorMap tmBlo, Args p) {
  using SM = Smem<BN, ST>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + SM::STAGES * SM::STAGE_BYTES);
  uint64_t* full_bar = bars;                     // TMA landed
  uint64_t* split_bar = bars + SM::STAGES;       // operand split done
  uint64_t* empty_bar = bars + 2 * SM::STAGES;   // MMAs that read the stage retired
  uint64_t* tmem_full_bar = bars + 3 * SM::STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * SM::STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * BM;
  const int zz = blockIdx.y;
  const int z = zz / p.ksplit;  // output slice
  const int nb = blockIdx.z;    // 128-column block of wide outputs
  const int total_kb = p.S * p.kb_per_slice;
  const int kb0 = (zz - z * p.ksplit) * p.kb_per_split;            // first k-block of this split
  const int num_kb = min(p.kb_per_split, total_kb - kb0);           // k-blocks of this split

  if (threadIdx.x == 0) {
    for (int s = 0; s < SM::STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&split_bar[s], 128);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {  // TMEM: BN fp32 accumulator columns x 128 lanes
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "n"(BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int stage = kb % SM::STAGES, phase = (kb / SM::STAGES) & 1;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* st = base + stage * SM::STAGE_BYTES;
        const int s = (kb0 + kb) / p.kb_per_slice, k0 = (kb0 + kb - s * p.kb_per_slice) * BK;
        mbar_expect_tx(&full_bar[stage], A_TILE_BYTES + 2 * SM::B_TILE_BYTES);
        if (s == 0)
          tma_load_2d(st, &tmA0, &full_bar[stage], k0, m0);
        else
          tma_load_2d(st, &tmA1, &full_bar[stage], k0, (s - 1) * p.rows_slice1 + m0);
        const int brow = (z * p.S + s) * p.b_rows_slice + nb * BN;
        tma_load_2d(st + 2 * A_TILE_BYTES, &tmBhi, &full_bar[stage], k0, brow);
        tma_load_2d(st + 2 * A_TILE_BYTES + SM::B_TILE_BYTES, &tmBlo, &full_bar[stage], k0, brow);
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0) {
      // instruction descriptor: D = f32, A = B = tf32, both K-major, N = BN, M = 128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int stage = kb % SM::STAGES, phase = (kb / SM::STAGES) & 1;
        mbar_wait(&split_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(base + stage * SM::STAGE_BYTES);
        const uint32_t sa_lo = sa + A_TILE_BYTES;
        const uint32_t sb_hi = sa + 2 * A_TILE_BYTES, sb_lo = sb_hi + SM::B_TILE_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint32_t koff = k * UMMA_K * 4;  // bytes inside the 128-byte swizzle row
          const uint64_t a_hi = make_desc(sa + koff), a_lo = make_desc(sa_lo + koff);
          const uint64_t b_hi = make_desc(sb_hi + koff), b_lo = make_desc(sb_lo + koff);
          umma_tf32(tmem_base, a_lo, b_hi, idesc, (kb | k) != 0);
          umma_tf32(tmem_base, a_hi, b_lo, idesc, 1);
          umma_tf32(tmem_base, a_hi, b_hi, idesc, 1);
        }
        umma_commit(&empty_bar[stage]);  // frees the stage once these MMAs have read it
      }
      umma_commit(tmem_full_bar);
    }
  } else {
    // ================= operand splitter, then epilogue =================
    const int t = threadIdx.x - 64;  // 0..127
    for (int kb = 0; kb < num_kb; ++kb) {
      const int stage = kb % SM::STAGES, phase = (kb / SM::STAGES) & 1;
      mbar_wait(&full_bar[stage], phase);
      float4* a = reinterpret_cast<float4*>(base + stage * SM::STAGE_BYTES);
      float4* alo = reinterpret_cast<float4*>(base + stage * SM::STAGE_BYTES + A_TILE_BYTES);
#pragma unroll
      for (int i = 0; i < A_TILE_BYTES / 16 / 128; ++i) {
        const int idx = t + 128 * i;
        const float4 v = a[idx];
        float4 hi, lo;
        hi.x = tf32_rn(v.x);
        hi.y = tf32_rn(v.y);
        hi.z = tf32_rn(v.z);
        hi.w = tf32_rn(v.w);
        lo.x = tf32_rn(v.x - hi.x);
        lo.y = tf32_rn(v.y - hi.y);
        lo.z = tf32_rn(v.z - hi.z);
        lo.w = tf32_rn(v.w - hi.w);
        a[idx] = hi;
        alo[idx] = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic-proxy writes -> tensor core reads
      mbar_arrive(&split_bar[stage]);
    }
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const int q = warp & 3;  // TMEM lane quarter this warp may access: tile rows 32q .. 32q+31
    // Each thread owns one accumulator row.  32-column chunks are staged through shared memory (the
    // pipeline stages are free now) so that the global stores are row-contiguous 128-byte segments.
    float* stg = reinterpret_cast<float*>(base) + (warp - 2) * (32 * 36);
    float* __restrict__ Cz = p.C + (long long)zz * p.sliceC;
    const bool vec_ok = ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(Cz) & 15) == 0);
    float loss_acc = 0.f;
    // bias has been added; accumulate / activation / loss epilogue of one element
    // y, w: this element's target and weight (fused loss epilogue only), fetched by the caller for a whole 32-column
    // chunk at once: one load per element issued right where it is used made every one of a thread's 32 row visits
    // wait for its own HBM round trip (the [B, 2 n_tasks] targets and weights are read exactly once: 63 us for the
    // ToxCast logits, the longest kernel of the step)
    auto finish = [&](float x, float old, float y, float w) -> float {
      if (p.accumulate) x += old;
      if (p.bce_y) {
        if constexpr (L2) {
          // weighted L2, tf.square(tf.mul(tf.sub(x, t), w)): loss and its gradient
          const float d = w * (x - y);
          loss_acc += d * d;
          return 2.f * w * d * p.bce_scale;
        } else {
          // weighted sigmoid cross-entropy with logits (multitask_classifier.py:41-44): loss and its gradient
          loss_acc += w * (fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x))));
          return w * (1.f / (1.f + expf(-x)) - y) * p.bce_scale;
        }
      }
      return (p.act == AGCN_ACT_RELU) ? fmaxf(x, 0.f) : x;
    };
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (nb * BN + c0 >= p.N) break;
      uint32_t v[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
          "%29,%30,%31}, [%32];\n"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
            "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
            "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
            "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
      for (int u = 0; u < 8; ++u)
        *reinterpret_cast<float4*>(&stg[lane * 36 + 4 * u]) =
            make_float4(__uint_as_float(v[4 * u]), __uint_as_float(v[4 * u + 1]), __uint_as_float(v[4 * u + 2]),
                        __uint_as_float(v[4 * u + 3]));
      __syncwarp();
      const int cc = nb * BN + c0 + 4 * (lane & 7);  // first of this lane's 4 output columns
      const float sc = p.scale ? __ldg(p.scale) : 1.f;
      float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (p.bias) {
        if (cc + 0 < p.N) bv.x = p.bias[cc + 0];
        if (cc + 1 < p.N) bv.y = p.bias[cc + 1];
        if (cc + 2 < p.N) bv.z = p.bias[cc + 2];
        if (cc + 3 < p.N) bv.w = p.bias[cc + 3];
      }
      // targets / weights of my 8 rows x 4 columns of this chunk, all 64 loads in flight together
      float yv[8][4], wv[8][4];
      if (p.bce_y) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int m = m0 + q * 32 + 4 * i + (lane >> 3);
          const long long bo = (long long)m * p.bce_ld + cc;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool ok = m < p.M && cc + e < p.N;
            yv[i][e] = ok ? __ldg(p.bce_y + bo + e) : 0.f;
            wv[i][e] = ok ? __ldg(p.bce_w + bo + e) : 0.f;
          }
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = 4 * i + (lane >> 3);
        const int m = m0 + q * 32 + r;
        float4 o = *reinterpret_cast<const float4*>(&stg[r * 36 + 4 * (lane & 7)]);
        if (m < p.M && cc < p.N) {
          const long long off = (long long)m * p.ldc + cc;
          float* dst = Cz + off;
          o.x = o.x * sc + bv.x; o.y = o.y * sc + bv.y; o.z = o.z * sc + bv.z; o.w = o.w * sc + bv.w;
          if constexpr (PROB) {
            // loss terms in the order of the training epilogue (the gradient finish() returns is dropped), then
            // probs[2t + c] = 1 / (1 + exp(x[2t + 1 - c] - x[2t + c]))  (L2: the values x)
            const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (cc + e < p.N) (void)finish(ov[e], 0.f, yv[i][e], wv[i][e]);
            const float4 pr = L2 ? o
                                 : make_float4(1.f / (1.f + expf(o.y - o.x)), 1.f / (1.f + expf(o.x - o.y)),
                                               1.f / (1.f + expf(o.w - o.z)), 1.f / (1.f + expf(o.z - o.w)));
            if (vec_ok && cc + 3 < p.N) {
              *reinterpret_cast<float4*>(dst) = pr;
            } else {
              const float pv[4] = {pr.x, pr.y, pr.z, pr.w};
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (cc + e < p.N) dst[e] = pv[e];
            }
          } else if (vec_ok && cc + 3 < p.N) {
            float4 old = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.accumulate) old = *reinterpret_cast<const float4*>(dst);
            o.x = finish(o.x, old.x, yv[i][0], wv[i][0]); o.y = finish(o.y, old.y, yv[i][1], wv[i][1]);
            o.z = finish(o.z, old.z, yv[i][2], wv[i][2]); o.w = finish(o.w, old.w, yv[i][3], wv[i][3]);
            *reinterpret_cast<float4*>(dst) = o;
          } else {
            const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              if (cc + e < p.N) dst[e] = finish(ov[e], p.accumulate ? dst[e] : 0.f, yv[i][e], wv[i][e]);
            }
          }
        }
      }
      __syncwarp();
    }
    if (p.loss_part) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, o);
      const int cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
      if (lane == 0) p.loss_part[cta * 4 + (warp - 2)] = loss_acc * p.bce_scale;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(BN) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// TN contraction over the node dimension on the tensor cores:
//     P_chunk[(f*S + s)*N + c] = sum_{r in chunk} A_s[r, f] * D[r, c]
// Both operands are row-major node matrices, i.e. MN-major for the MMA (the contraction index r is the
// slow one).  MN-major TF32 operands must use the "128B swizzle, 32B atom" shared-memory layout (UMMA layout
// type 1 / CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): TMA brings 32-row x 32-column boxes, four rows form one
// 512-byte swizzle atom (stride byte offset), a k-step of 8 rows is 1024 bytes, and the 32-column groups of
// one operand are 4096 bytes apart (leading byte offset).
// Both operands are activations, so both are split hi/lo in shared memory.
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)(4096 >> 4) << 16;  // leading byte offset: next group of 32 M/N elements
  d |= (uint64_t)(512 >> 4) << 32;   // stride byte offset: next group of 4 K rows
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;            // SWIZZLE_128B_BASE32B
  return d;
}

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

struct TnArgs {
  int M;        // rows contracted (nodes)
  int Kd;       // columns of A_s = rows of the result (<= 128)
  int N;        // columns of D
  int S;
  int kb_per_chunk;
  float* partial;   // [chunks][Kd*S*N]
};

template <int BN>
struct SmemTn {
  static constexpr int A_BYTES = 128 * BK * 4;   // 4 boxes of 32 rows x 128 bytes
  static constexpr int B_BYTES = BN * BK * 4;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr int STAGES = (BN <= 64) ? 4 : 3;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256;
};

template <int BN>
__global__ void __launch_bounds__(192, 1)
tc_gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                  const __grid_constant__ CUtensorMap tmD, TnArgs p) {
  using SM = SmemTn<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + SM::STAGES * SM::STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* split_bar = bars + SM::STAGES;
  uint64_t* empty_bar = bars + 2 * SM::STAGES;
  uint64_t* tmem_full_bar = bars + 3 * SM::STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * SM::STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunk = blockIdx.x, s = blockIdx.y, nb = blockIdx.z;
  const int total_kb = (p.M + BK - 1) / BK;
  const int kb_begin = chunk * p.kb_per_chunk;
  const int num_kb = min(p.kb_per_chunk, total_kb - kb_begin);
  const int a_boxes = (p.Kd + 31) / 32;                       // 32-column groups of A that exist
  const int b_boxes = min(BN / 32, (p.N - nb * BN + 31) / 32);  // of this column block of D

  // boxes that are never loaded stay zero for the whole kernel
  for (int i = threadIdx.x; i < SM::STAGES * SM::STAGE_BYTES / 16; i += blockDim.x)
    reinterpret_cast<float4*>(base)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (threadIdx.x == 0) {
    for (int i = 0; i < SM::STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&split_bar[i], 128);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "n"(BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // zero fill above vs. TMA / tensor-core reads
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int stage = kb % SM::STAGES, phase = (kb / SM::STAGES) & 1;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* st = base + stage * SM::STAGE_BYTES;
        const int r0 = (kb_begin + kb) * BK;
        mbar_expect_tx(&full_bar[stage], (a_boxes + b_boxes) * 4096);
        for (int b = 0; b < a_boxes; ++b) {
          if (s == 0)
            tma_load_3d(st + b * 4096, &tmA0, &full_bar[stage], 32 * b, r0, 0);
          else
            tma_load_3d(st + b * 4096, &tmA1, &full_bar[stage], 32 * b, r0, s - 1);
        }
        for (int b = 0; b < b_boxes; ++b)
          tma_load_3d(st + 2 * SM::A_BYTES + b * 4096, &tmD, &full_bar[stage], nb * BN + 32 * b, r0, 0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // D = f32, A = B = tf32, both MN-major, N = BN, M = 128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      for (int kb = 0; kb < num_kb; ++kb) {
        const int stage = kb % SM::STAGES, phase = (kb / SM::STAGES) & 1;
        mbar_wait(&split_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(base + stage * SM::STAGE_BYTES);
        const uint32_t sa_lo = sa + SM::A_BYTES;
        const uint32_t sb = sa + 2 * SM::A_BYTES, sb_lo = sb + SM::B_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k) {
          const uint32_t koff = k * 1024;  // 8 contraction rows = one swizzle atom
          const uint64_t a_hi = make_desc_mn(sa + koff), a_lo = make_desc_mn(sa_lo + koff);
          const uint64_t b_hi = make_desc_mn(sb + koff), b_lo = make_desc_mn(sb_lo + koff);
          umma_tf32(tmem_base, a_lo, b_hi, idesc, (kb | k) != 0);
          umma_tf32(tmem_base, a_hi, b_lo, idesc, 1);
          umma_tf32(tmem_base, a_hi, b_hi, idesc, 1);
        }
        umma_commit(&empty_bar[stage]);
      }
      umma_commit(tmem_full_bar);
    }
  } else {
    const int t = threadIdx.x - 64;
    for (int kb = 0; kb < num_kb; ++kb) {
      const int stage = kb % SM::STAGES, phase = (kb / SM::STAGES) & 1;
      mbar_wait(&full_bar[stage], phase);
      uint8_t* st = base + stage * SM::STAGE_BYTES;
      auto split = [&](float4* hi_p, float4* lo_p, int n16) {
        for (int idx = t; idx < n16; idx += 128) {
          const float4 v = hi_p[idx];
          float4 hi, lo;
          hi.x = tf32_rn(v.x);
          hi.y = tf32_rn(v.y);
          hi.z = tf32_rn(v.z);
          hi.w = tf32_rn(v.w);
          lo.x = tf32_rn(v.x - hi.x);
          lo.y = tf32_rn(v.y - hi.y);
          lo.z = tf32_rn(v.z - hi.z);
          lo.w = tf32_rn(v.w - hi.w);
          hi_p[idx] = hi;
          lo_p[idx] = lo;
        }
      };
      split(reinterpret_cast<float4*>(st), reinterpret_cast<float4*>(st + SM::A_BYTES), a_boxes * 256);
      split(reinterpret_cast<float4*>(st + 2 * SM::A_BYTES),
            reinterpret_cast<float4*>(st + 2 * SM::A_BYTES + SM::B_BYTES), b_boxes * 256);
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      mbar_arrive(&split_bar[stage]);
    }
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const int q = warp & 3;
    float* stg = reinterpret_cast<float*>(base) + (warp - 2) * (32 * 36);
    float* __restrict__ P = p.partial + (long long)chunk * p.Kd * p.S * p.N;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      if (nb * BN + c0 >= p.N) break;
      uint32_t v[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,"
          "%29,%30,%31}, [%32];\n"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
            "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
            "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
            "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
          : "r"(taddr));
      asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
      for (int u = 0; u < 8; ++u)
        *reinterpret_cast<float4*>(&stg[lane * 36 + 4 * u]) =
            make_float4(__uint_as_float(v[4 * u]), __uint_as_float(v[4 * u + 1]), __uint_as_float(v[4 * u + 2]),
                        __uint_as_float(v[4 * u + 3]));
      __syncwarp();
      const int cc = nb * BN + c0 + 4 * (lane & 7);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = 4 * i + (lane >> 3);
        const int f = q * 32 + r;  // result row = column of A_s
        if (f < p.Kd && cc < p.N) {
          const float4 o = *reinterpret_cast<const float4*>(&stg[r * 36 + 4 * (lane & 7)]);
          float* dst = P + ((long long)f * p.S + s) * p.N + cc;
          if ((p.N & 3) == 0) {
            *reinterpret_cast<float4*>(dst) = o;
          } else {
            const float ov[4] = {o.x, o.y, o.z, o.w};
            for (int e = 0; e < 4; ++e)
              if (cc + e < p.N) dst[e] = ov[e];
          }
        }
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(BN) : "memory");
  }
}

// B prep: out_{hi,lo}[(slice*Npad + n)*Kd + k] = split(src[n*sn + k*sk + slice*ss]),  zero rows for n >= N
// (Kp = Kd rounded up to 4 is the row pitch: TMA needs 16-byte row strides; the pad columns are zero)
__global__ void split_b_kernel(const float* __restrict__ src, long long sn, long long sk, long long ss, int N, int Npad,
                               int Kd, int Kp, int slices, float* __restrict__ hi, float* __restrict__ lo) {
  const long long total = (long long)slices * Npad * Kp;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(e % Kp);
    const long long r = e / Kp;
    const int n = (int)(r % Npad), sl = (int)(r / Npad);
    float x = 0.f;
    if (n < N && k < Kd) x = src[n * sn + k * sk + sl * ss];
    const float h = tf32_rn(x);
    hi[e] = h;
    lo[e] = tf32_rn(x - h);
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

// 2-D fp32 row-major [rows, cols] with leading dimension ld; box = 32 columns x box_rows, 128-byte swizzle
static int make_map(CUtensorMap* map, const float* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return AGCN_ERR_CUDA;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld * sizeof(float)};
  cuuint32_t box[2] = {(cuuint32_t)BK, box_rows};
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

// 3-D fp32 [slices, rows, cols] (cols contiguous, row pitch ld, slice pitch slice_elems); box = 32 x 32 x 1
static int make_map3(CUtensorMap* map, const float* ptr, uint64_t slices, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint64_t slice_elems) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return AGCN_ERR_CUDA;
  }
  cuuint64_t gdim[3] = {cols, rows, slices};
  cuuint64_t gstride[2] = {ld * sizeof(float), slice_elems * sizeof(float)};
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (3d) failed with code " + std::to_string((int)r));
    return AGCN_ERR_CUDA;
  }
  return AGCN_OK;
}

}  // namespace tc

__global__ void reduce_chunks_kernel(const float* __restrict__ partial, float* __restrict__ out, long long elems,
                                     int chunks);

static int tc_npad(int N) { return N <= 64 ? 64 : (N + 127) / 128 * 128; }
static int tc_kpitch(int Kd) { return (Kd + 3) & ~3; }

bool tc_gemm_supported(const GemmArgs& a) {
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (a.M < 1 || a.Kd < 32) return false;
  if (a.S > 1 && a.Kd % 4 != 0) return false;  // stacked slices share one tensor map
  if (a.lda0 % 4 != 0 || !al16(a.A0)) return false;
  if (a.S > 1 && (a.lda1 % 4 != 0 || !al16(a.A1) || a.sliceA1 % a.lda1 != 0)) return false;
  if (a.S > 1 && a.lda1 != a.Kd) return false;  // slices are stacked as one [(S-1)*rows, Kd] matrix
  return true;
}

// The fused-loss logits product (M = batch, N = 2 n_tasks) has fewer 128-column tiles than SMs and a long epilogue per
// tile: 64-column tiles, two stages, two CTAs per SM put twice as many CTAs to work at once
// (ToxCast head, 1024 x 1234 x 256: 55 us with 80 CTAs of 128 columns).  The decision depends on bce_y / prob only,
// not on which loss (l2) they carry: a head's training and prediction products tile alike, so their loss terms are
// added up in the same order.
static bool tc_gemm_narrow2(const GemmArgs& a) {
  const int Npad = tc_npad(a.N);
  if (!(a.bce_y || a.prob) || Npad <= 64) return false;
  const int tiles128 = ((a.M + tc::BM - 1) / tc::BM) * a.Z * (Npad / 128);
  return tiles128 < 148;
}

int tc_gemm_loss_parts(const GemmArgs& a) {
  const int Npad = tc_npad(a.N), BN = (Npad <= 64 || tc_gemm_narrow2(a)) ? 64 : 128;
  return 4 * ((a.M + tc::BM - 1) / tc::BM) * a.Z * (Npad / BN);
}

// split-K for long contractions with few output tiles (plain outputs only): chunk ks of the contraction writes its raw
// partial sums to split_k_partial + ks * M * ldc, and reduce_chunks_kernel adds them in the order ks = 0, 1, ...
static void tc_gemm_split(const GemmArgs& a, int* ksplit, int* kb_per_split) {
  using namespace tc;
  const int Npad = tc_npad(a.N), BN = (Npad <= 64 || tc_gemm_narrow2(a)) ? 64 : 128;
  const int total_kb = a.S * ((a.Kd + BK - 1) / BK);
  const int out_tiles = ((a.M + BM - 1) / BM) * a.Z * (Npad / BN);
  int k = 1;
  if (a.split_k_partial && !a.bias && !a.scale && a.act == AGCN_ACT_LINEAR && !a.accumulate && !a.bce_y && !a.prob &&
      a.ldc == a.N && a.Z == 1 && total_kb >= 16 && out_tiles < 74)
    k = std::min(std::min(8, total_kb / 4), std::max(1, 148 / out_tiles));
  *kb_per_split = (total_kb + k - 1) / k;
  *ksplit = (total_kb + *kb_per_split - 1) / *kb_per_split;
}

int tc_gemm_ksplit(const GemmArgs& a) {
  int ksplit, per;
  tc_gemm_split(a, &ksplit, &per);
  return ksplit;
}

size_t tc_gemm_scratch_floats(int N, int Kd, int S, int Z) { return 2 * (size_t)Z * S * tc_npad(N) * tc_kpitch(Kd); }

// Rearranges the parameter operand B to [slice][Npad][Kd] (K-major) and splits it into hi / lo TF32 halves.
// It depends on the parameters only, so callers run it on a side stream (or once per forward/backward pair).
int tc_gemm_split_b(const GemmArgs& a, float* scratch, cudaStream_t st) {
  using namespace tc;
  // B element (slice, n, k): row-major [Kd, N] (ldb) or, transposed, [N, Kd]
  const long long sn = a.transB ? a.ldb : 1, sk = a.transB ? 1 : a.ldb, ss = a.sliceB;
  const int Npad = tc_npad(a.N), Kp = tc_kpitch(a.Kd);
  const int slices = a.Z * a.S;
  float* Bhi = scratch;
  float* Blo = scratch + (size_t)slices * Npad * Kp;
  const long long total = (long long)slices * Npad * Kp;
  const int blocks = (int)std::min<long long>((total + 255) / 256, 1184);
  split_b_kernel<<<blocks, 256, 0, st>>>(a.B, sn, sk, ss, a.N, Npad, a.Kd, Kp, slices, Bhi, Blo);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

template <int BN, int ST, bool PROB, bool L2>
static void launch_tc_gemm_kernel(dim3 grid, const CUtensorMap& mA0, const CUtensorMap& mA1, const CUtensorMap& mBhi,
                                  const CUtensorMap& mBlo, const tc::Args& p, cudaStream_t st) {
  using namespace tc;
  static std::once_flag once;
  std::call_once(once, [] {
    cudaFuncSetAttribute(tc_gemm_kernel<BN, ST, PROB, L2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         Smem<BN, ST>::TOTAL);
  });
  ProfScope prof(L2 ? (PROB ? "tc::tc_gemm_kernel<l2,prob>" : "tc::tc_gemm_kernel<l2>")
                    : (PROB ? "tc::tc_gemm_kernel<prob>" : "tc::tc_gemm_kernel"),
                 st);
  tc_gemm_kernel<BN, ST, PROB, L2><<<grid, 192, Smem<BN, ST>::TOTAL, st>>>(mA0, mA1, mBhi, mBlo, p);
}

template <bool PROB, bool L2>
static void launch_tc_gemm(bool narrow2, int BN, dim3 grid, const CUtensorMap& mA0, const CUtensorMap& mA1,
                           const CUtensorMap& mBhi, const CUtensorMap& mBlo, const tc::Args& p, cudaStream_t st) {
  if (narrow2)
    launch_tc_gemm_kernel<64, 2, PROB, L2>(grid, mA0, mA1, mBhi, mBlo, p, st);
  else if (BN == 64)
    launch_tc_gemm_kernel<64, 0, PROB, L2>(grid, mA0, mA1, mBhi, mBlo, p, st);
  else
    launch_tc_gemm_kernel<128, 0, PROB, L2>(grid, mA0, mA1, mBhi, mBlo, p, st);
}

// scratch holds the hi / lo copies of B written by tc_gemm_split_b (tc_gemm_scratch_floats floats).
int tc_gemm(const GemmArgs& a, const float* scratch, cudaStream_t st) {
  using namespace tc;
  const int Npad = tc_npad(a.N), Kp = tc_kpitch(a.Kd);
  const int slices = a.Z * a.S;
  const float* Bhi = scratch;
  const float* Blo = scratch + (size_t)slices * Npad * Kp;
  CUtensorMap mA0, mA1, mBhi, mBlo;
  int rc;
  if ((rc = make_map(&mA0, a.A0, (uint64_t)a.M, (uint64_t)a.Kd, (uint64_t)a.lda0, BM))) return rc;
  const int rows_slice1 = a.S > 1 ? (int)(a.sliceA1 / a.lda1) : 0;
  if (a.S > 1) {
    if ((rc = make_map(&mA1, a.A1, (uint64_t)(a.S - 2) * rows_slice1 + a.M, (uint64_t)a.Kd, (uint64_t)a.lda1, BM)))
      return rc;
  } else {
    mA1 = mA0;
  }
  const bool narrow2 = tc_gemm_narrow2(a);
  const int BN = (Npad <= 64 || narrow2) ? 64 : 128;
  if ((rc = make_map(&mBhi, Bhi, (uint64_t)slices * Npad, (uint64_t)a.Kd, (uint64_t)Kp, BN))) return rc;
  if ((rc = make_map(&mBlo, Blo, (uint64_t)slices * Npad, (uint64_t)a.Kd, (uint64_t)Kp, BN))) return rc;
  Args p;
  p.M = a.M; p.N = a.N; p.Kd = a.Kd; p.S = a.S;
  p.kb_per_slice = (a.Kd + BK - 1) / BK;
  tc_gemm_split(a, &p.ksplit, &p.kb_per_split);
  const int ksplit = p.ksplit;
  p.rows_slice1 = rows_slice1;
  p.b_rows_slice = Npad;
  p.C = a.C; p.ldc = a.ldc; p.sliceC = a.sliceC;
  if (ksplit > 1) {
    p.C = a.split_k_partial;
    p.sliceC = (long long)a.M * a.ldc;
  }
  p.bias = a.bias; p.scale = a.scale; p.act = a.act; p.accumulate = a.accumulate;
  p.bce_y = a.bce_y; p.bce_w = a.bce_w; p.bce_scale = a.bce_scale; p.loss_part = a.loss_part;
  p.bce_ld = a.bce_ld > 0 ? a.bce_ld : a.ldc;
  dim3 grid((a.M + BM - 1) / BM, a.Z * ksplit, Npad / BN);
  if (a.l2 && a.prob)
    launch_tc_gemm<true, true>(narrow2, BN, grid, mA0, mA1, mBhi, mBlo, p, st);
  else if (a.l2)
    launch_tc_gemm<false, true>(narrow2, BN, grid, mA0, mA1, mBhi, mBlo, p, st);
  else if (a.prob)
    launch_tc_gemm<true, false>(narrow2, BN, grid, mA0, mA1, mBhi, mBlo, p, st);
  else
    launch_tc_gemm<false, false>(narrow2, BN, grid, mA0, mA1, mBhi, mBlo, p, st);
  AGCN_LAUNCH_CHECK();
  if (ksplit > 1 && !a.split_k_raw) {
    const long long elems = (long long)a.M * a.ldc;
    reduce_chunks_kernel<<<(unsigned)((elems + 255) / 256), 256, 0, st>>>(a.split_k_partial, a.C, elems, ksplit);
    AGCN_LAUNCH_CHECK();
  }
  return AGCN_OK;
}

}  // namespace agcn

namespace agcn {

bool tc_gemm_tn_supported(const GemmTNArgs& a) {
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (a.M < 32 || a.Kd > 128 || a.Kd % 4 != 0 || a.N % 4 != 0) return false;
  if (a.lda0 % 4 != 0 || a.ldd % 4 != 0 || !al16(a.A0) || !al16(a.D)) return false;
  if (a.S > 1 && (a.lda1 % 4 != 0 || !al16(a.A1) || a.sliceA1 % 4 != 0)) return false;
  return true;
}

static void tn_chunks(const GemmTNArgs& a, int* chunks, int* kb_per_chunk) {
  const int total_kb = (a.M + tc::BK - 1) / tc::BK;
  const int nblk = (a.N + 127) / 128;
  int want = std::max(1, 148 / std::max(1, a.S * nblk));
  int per = std::max(4, (total_kb + want - 1) / want);
  *kb_per_chunk = per;
  *chunks = (total_kb + per - 1) / per;
}

size_t tc_gemm_tn_partial_floats(const GemmTNArgs& a) {
  int chunks, per;
  tn_chunks(a, &chunks, &per);
  return (size_t)chunks * a.Kd * a.S * a.N;
}

__global__ void reduce_chunks_kernel(const float* __restrict__ partial, float* __restrict__ out, long long elems,
                                     int chunks) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= elems) return;
  float s = 0.f;
  for (int k = 0; k < chunks; ++k) s += partial[(long long)k * elems + e];
  out[e] = s;
}

int tc_gemm_tn(const GemmTNArgs& a, cudaStream_t st) {
  using namespace tc;
  if (!tc_gemm_tn_supported(a)) {
    set_error("gemm_tn: shape not supported by the tensor-core kernel");
    return AGCN_ERR_INVALID;
  }
  int chunks, per;
  tn_chunks(a, &chunks, &per);
  CUtensorMap mA0, mA1, mD;
  int rc;
  if ((rc = make_map3(&mA0, a.A0, 1, (uint64_t)a.M, (uint64_t)a.Kd, (uint64_t)a.lda0, (uint64_t)a.M * a.lda0))) return rc;
  if (a.S > 1) {
    if ((rc = make_map3(&mA1, a.A1, (uint64_t)(a.S - 1), (uint64_t)a.M, (uint64_t)a.Kd, (uint64_t)a.lda1,
                        (uint64_t)a.sliceA1)))
      return rc;
  } else {
    mA1 = mA0;
  }
  if ((rc = make_map3(&mD, a.D, 1, (uint64_t)a.M, (uint64_t)a.N, (uint64_t)a.ldd, (uint64_t)a.M * a.ldd))) return rc;
  TnArgs p;
  p.M = a.M; p.Kd = a.Kd; p.N = a.N; p.S = a.S;
  p.kb_per_chunk = per;
  p.partial = a.partial;
  const int BN = a.N <= 64 ? 64 : 128;
  dim3 grid(chunks, a.S, (a.N + BN - 1) / BN);
  static std::once_flag once64, once128;
  if (BN == 64) {
    std::call_once(once64, [] {
      cudaFuncSetAttribute(tc_gemm_tn_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemTn<64>::TOTAL);
    });
    {
      ProfScope prof("tc::tc_gemm_tn_kernel", st);
      tc_gemm_tn_kernel<64><<<grid, 192, SmemTn<64>::TOTAL, st>>>(mA0, mA1, mD, p);
    }
  } else {
    std::call_once(once128, [] {
      cudaFuncSetAttribute(tc_gemm_tn_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemTn<128>::TOTAL);
    });
    {
      ProfScope prof("tc::tc_gemm_tn_kernel", st);
      tc_gemm_tn_kernel<128><<<grid, 192, SmemTn<128>::TOTAL, st>>>(mA0, mA1, mD, p);
    }
  }
  AGCN_LAUNCH_CHECK();
  const long long elems = (long long)a.Kd * a.S * a.N;
  reduce_chunks_kernel<<<(unsigned)((elems + 255) / 256), 256, 0, st>>>(a.partial, a.out, elems, chunks);
  AGCN_LAUNCH_CHECK();
  return AGCN_OK;
}

}  // namespace agcn
